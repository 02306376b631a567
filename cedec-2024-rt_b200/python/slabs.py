"""slabs — row-slab partition of a frame over the GPUs of one node and the halo exchange it needs.

The reference is single-GPU; this is new host logic (SURVEY.md section 8e).  Every kernel is per-pixel independent
except spatial_resampling, which reads the reservoirs and the sky/emissive class of up to 5 neighbours within
+-86.4 px (sample_2d_gaussian with rv0 >= 2^-23 and radius/1.96, examples/10_restir_di/10_restir_di.cu:309-313), so

  * rank r computes image rows yi in [y0, y1) (crt_set_row_range); buffers are full-size and indices global;
  * before every spatial pass each rank sends the HALO = 87 boundary rows of the pass's input reservoirs to its
    slab neighbours and receives theirs into the same global positions; in drop-in mode the same happens once per
    frame for the Visibility rows the neighbour rejection reads (in fused mode the sky/emissive marker travels inside
    the reservoir records themselves, csrc/restir_fast.cuh: kSkipBit).

Nothing here touches pixel data itself: the functions compute byte ranges of bottom-up buffers
(pixel_idx = xi + (H - yi - 1) * W, 10_restir_di.cu:18-20) and issue torch.distributed P2P ops on them, so the same
code runs over NCCL on GPU tensors (bench.py) and over gloo on CPU tensors (tests/test_slabs.py).
"""

import math

HALO = 87  # rows the direct-store (p2p) path mirrors: |neighbour offset| <= 86.4 px at the reference's radius 30 (csrc: kHaloRows)


def halo_rows(radius):
    """rows a spatial pass can reach beyond its own: the neighbour offset is radius / 1.96 * r * cos|sin(phi) with
    r = sqrt(-2 ln rv0) and rv0 >= 2^-23 (rv0 = 0 gives an infinite offset, which is skipped as off-screen), truncated
    towards zero (10_restir_di.cu:309-313, reservoir.hpp:89-95) — which rounds the reach *up* on the side of smaller
    coordinates: floor(offset) + 1 rows; the factor covers the float rounding of the product"""
    return int(math.floor(abs(float(radius)) / 1.96 * math.sqrt(-2.0 * math.log(2.0 ** -23)) * (1.0 + 1e-5))) + 1


def slab_rows(H, world, rank, align=8):
    """rows [y0, y1) of rank `rank`: equal shares rounded to multiples of `align` rows (the kernels' tile height)"""
    edges = [((H * r // world) + align - 1) // align * align for r in range(world)] + [H]
    edges[0] = 0
    edges = [min(e, H) for e in edges]
    return edges[rank], edges[rank + 1]


def weighted_slab_rows(row_cost, world, align=8, min_rows=0):
    """slab edges that balance a per-row cost estimate (e.g. measured slab times spread over their rows) instead
    of row counts; every slab gets at least `min_rows` rows; returns the list of world + 1 edges"""
    H = len(row_cost)
    total = float(sum(row_cost))
    edges, acc, r = [0], 0.0, 1
    for y, c in enumerate(row_cost):
        acc += c
        while r < world and acc >= total * r / world:
            e = min(H, max(edges[-1] + min_rows, (y + 1 + align - 1) // align * align))
            edges.append(e)
            r += 1
    while len(edges) < world:
        edges.append(H)
    edges.append(H)
    # leave room for the slabs below: the last ones must keep min_rows too
    for i in range(world - 1, 0, -1):
        edges[i] = min(edges[i], edges[i + 1] - min_rows)
    for i in range(1, world):
        edges[i] = max(edges[i], edges[i - 1] + min_rows) // align * align
    return edges


def rebalance(edges, slab_ms, align=8, min_rows=0):
    """new edges from the measured compute time of every slab: the cost of a slab is spread evenly over its rows"""
    H, world = edges[-1], len(edges) - 1
    cost = [0.0] * H
    for r in range(world):
        rows = edges[r + 1] - edges[r]
        for y in range(edges[r], edges[r + 1]):
            cost[y] = slab_ms[r] / max(rows, 1)
    return weighted_slab_rows(cost, world, align, min_rows)


def halo_plan(H, edges, rank, halo=HALO):
    """[(peer, send_rows, recv_rows)]: the rows of mine every other rank's spatial pass can read, and the rows of
    theirs mine can.  With slabs taller than `halo` this is the two adjacent slabs; thin slabs reach further."""
    y0, y1 = edges[rank], edges[rank + 1]
    plan = []
    for peer in range(len(edges) - 1):
        if peer == rank:
            continue
        p0, p1 = edges[peer], edges[peer + 1]
        if p1 <= p0 or y1 <= y0:
            continue
        # rows of mine within `halo` of the peer's slab, and vice versa
        send = (max(y0, p0 - halo), min(y1, p1 + halo))
        recv = (max(p0, y0 - halo), min(p1, y1 + halo))
        if send[0] < send[1] and recv[0] < recv[1]:
            plan.append((peer, send, recv))
    return plan


def full_plan(H, edges, rank):
    """the halo plan with an unbounded reach: every rank sends all its rows to every other rank and receives all of
    theirs (the history gather of temporal reprojection, SlabRenderer.gather_history)"""
    return halo_plan(H, edges, rank, halo=H)


def row_byte_ranges(W, H, rows, layout):
    """byte ranges [(begin, end)] that image rows [a, b) occupy in a bottom-up buffer.
    layout: ("aos", elem_bytes) — one contiguous range; ("planes", [elem_bytes...]) — planar storage over W*H
    pixels, planes back to back in the order given (plane p starts where plane p-1 ends), as in
    csrc/restir_fast.cuh: soa_plane_offset."""
    a, b = rows
    first, last = (H - b) * W, (H - a) * W
    if layout[0] == "aos":
        e = layout[1]
        return [(first * e, last * e)]
    out, off = [], 0
    for e in layout[1]:
        out.append((off + first * e, off + last * e))
        off += e * W * H
    return out


SOA_RESERVOIR = ("planes", [32, 32, 8])  # csrc/restir_fast.cuh: SoaStore
AOS_RESERVOIR = ("aos", 76)
AOS_VISIBILITY = ("aos", 16)
CLASS_PLANE = ("aos", 1)


def exchange(dist, tensor, W, H, layout, plan):
    """send/receive the halo rows of one flat uint8 tensor (a full-size bottom-up buffer) according to `plan`;
    returns the bytes this rank sent"""
    if not plan:
        return 0
    ops, sent = [], 0
    for peer, send_rows, recv_rows in plan:
        for (s0, s1) in row_byte_ranges(W, H, send_rows, layout):
            ops.append(dist.P2POp(dist.isend, tensor[s0:s1], peer))
            sent += s1 - s0
        for (r0, r1) in row_byte_ranges(W, H, recv_rows, layout):
            ops.append(dist.P2POp(dist.irecv, tensor[r0:r1], peer))
    for req in dist.batch_isend_irecv(ops):
        req.wait()
    return sent


class CudaArrayView:
    """device memory owned by libcedecrt as a torch tensor (zero-copy, __cuda_array_interface__)"""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class SlabRenderer:
    """The frame loop over one GPU's row slab.  Buffers are full-size (pixel indices stay global) and are torch
    tensors, so that torch.distributed can move halo rows; kernels run through the C ABI on torch's stream."""

    def __init__(self, torch, dist, rank, world, tris, cam, W, H, fused=True, edges=None, options=None, p2p=True,
                 stream=None, share=None, connect=True, overlap=False, reproject=False):
        """p2p: in fused mode with more than one rank, exchange halo rows by direct peer stores (csrc/slab_p2p.cu,
        buffers shared through cudaIpc handles) instead of NCCL send/recv; needs slabs >= HALO rows, W % 16 == 0.
        stream: the torch stream this slab's kernels go to (default: the current one).  share: another SlabRenderer on
        the same GPU whose scene, light list and BVH this one uses instead of uploading and building its own.
        connect=False leaves the neighbour links to the caller (SlabGroup: slabs of one process are linked by plain
        pointers, `rank`/`world` then count slabs, not processes).  overlap: fused mode only — the frame's tail (resolve
        rays + tone mapping) runs on the context's second stream beside the next frame's head (crt_set_frame_overlap).
        reproject (extension, DESIGN.md section 11): temporal resampling looks the history up at the pixel the surface point
        had in the previous frame's camera (set_camera).  That pixel may lie in any slab — the displacement is bounded by the
        camera motion, not by the spatial halo — so before such a frame every rank receives every other rank's rows of the
        history (full_plan: the halo plan with an unbounded reach, over NCCL / gloo); the direct-store path mirrors halo
        rows only and is not used.
        reproject="surfaces": the same look-up with the previous frame's surfaces, which unbiased reuse weights need with a
        moving camera (cedecrt.RestirDI(reproject="surfaces")): two Visibility buffers alternate, and before a frame that
        looks the history up every rank also receives every other rank's rows of last frame's Visibility
        (crt_restir_set_previous_frame in fused mode, crt_temporal_resampling_reprojected_surfaces in drop-in mode).
        Under the reference's weights it renders what reproject=True renders.
        set_triangles() moves the geometry; with reprojection the next frame follows it (cedecrt.RestirDI.set_triangles:
        every rank holds the whole triangle array, so the previous one is local).
        With more than one slab the fused frame produces the G-buffer records of its halo rows itself
        (crt_restir_set_halo_surfaces), so that unbiased reuse weights (set_reuse_weights) run on every split of the frame;
        under the reference's weights that costs nothing."""
        import numpy as np

        import cedecrt

        self.torch, self.dist, self.rank, self.world, self.W, self.H = torch, dist, rank, world, W, H
        self.c = cedecrt
        self.options = options or cedecrt.Options(accumulate=1, use_temporal_resampling=1, use_spatial_resampling=1)
        # options the fused bodies do not cover (use_shadowed_target_function, an M bound past 2^29) make the crt_restir_*
        # calls take the per-kernel path on AoS buffers (kernels_fast.cu: fused()): the host must then exchange AoS
        # reservoir rows and Visibility rows, exactly as in drop-in mode
        self.fused = bool(fused and cedecrt.lib().crt_restir_is_fused(self.options))
        fused = self.fused
        self.halo = halo_rows(self.options.spatial_resampling_radius) if self.options.use_spatial_resampling else 0
        self.rt = cedecrt.Runtime(torch.cuda.current_device())
        self.stream = stream if stream is not None else torch.cuda.current_stream()
        assert self.stream.cuda_stream != 0, "bench needs a non-default torch stream"
        self.rt.set_stream(self.stream.cuda_stream)
        assert reproject in (False, True, "surfaces"), reproject
        self.reproject, self.prev_raygen = bool(reproject), None
        self.surfaces = reproject == "surfaces"
        # set_triangles: last frame's triangle array (allocated on the first move), passed on while `moved` is set
        self.t_tris_prev, self.prev_triangles, self.moved = None, None, False
        if self.reproject:
            p2p = False
        if self.fused and world > 1:
            self.rt.restir_set_halo_surfaces(True)
        self.overlap = bool(overlap and self.fused)
        self._tail = None
        if self.overlap:
            self.rt.set_frame_overlap(True)
            self._tail = torch.cuda.ExternalStream(self.rt.tail_stream())
        self.edges = edges if edges is not None else [slab_rows(H, world, r)[0] for r in range(world)] + [H]
        self.y0, self.y1 = self.edges[rank], self.edges[rank + 1]
        self.plan = halo_plan(H, self.edges, rank, self.halo) if world > 1 else []
        self.full_plan = full_plan(H, self.edges, rank) if world > 1 else []
        self.rt.set_row_range(self.y0, self.y1)
        self.eye = tuple(float(np.float32(v)) for v in cam[0])
        self.raygen = cedecrt.lookat(cam[0], cam[1], W, H)
        n = W * H
        dev = torch.device("cuda", torch.cuda.current_device())

        heights = [b - a for a, b in zip(self.edges, self.edges[1:])]
        # Direct peer stores need (a) slabs at least as tall as the mirrored band and a reach inside it (radius <= 30),
        # (b) at least two spatial passes: the only ordering between neighbours is one signal/wait per pass
        # (slab_p2p.cu), and with a single pass a fast neighbour could store frame f+1's temporal rows into this slab
        # while its pass of frame f still reads them.  Otherwise the rows travel by NCCL send/recv.
        passes_ok = (not self.options.use_spatial_resampling) or self.options.spatial_resampling_passes >= 2
        self.p2p = bool(p2p and fused and world > 1 and W % 16 == 0 and min(heights) >= HALO and self.halo <= HALO
                        and passes_ok)
        self._owned = []

        def tbuf(nbytes, dtype, count, zero=False, shared=False):
            if shared and self.p2p:  # cudaMalloc'ed by the library, so that it can be exported with cudaIpc
                b = self.rt.buffer(dtype, count)
                if zero:
                    b.zero()
                self._owned.append(b)
                return torch.as_tensor(CudaArrayView(b.ptr, nbytes), device=dev), b
            t = (torch.zeros if zero else torch.empty)(nbytes, dtype=torch.uint8, device=dev)
            return t, self.rt.wrap(t.data_ptr(), dtype, count)

        if share is not None:
            self.t_tris, self.t_lights, self.geom = share.t_tris, share.t_lights, share.geom
            self.n_tris, self.n_lights = share.n_tris, share.n_lights
            self.triangles = self.rt.wrap(self.t_tris.data_ptr(), cedecrt.TRIANGLE, self.n_tris)
            self.lights = self.rt.wrap(self.t_lights.data_ptr(), np.uint32, self.n_lights)
        else:
            self.t_tris = torch.from_numpy(tris.view(np.uint8).reshape(-1)).to(dev)
            self.triangles = self.rt.wrap(self.t_tris.data_ptr(), cedecrt.TRIANGLE, len(tris))
            lights = cedecrt.light_indices(tris)
            self.t_lights = torch.from_numpy(lights.view(np.uint8)).to(dev)
            self.lights = self.rt.wrap(self.t_lights.data_ptr(), np.uint32, len(lights))
            self.n_tris, self.n_lights = len(tris), len(lights)
            self.geom = self.rt.build_geometry(self.triangles)
        self.t_pix, self.pixels = tbuf(4 * n, np.uint8, 4 * n)
        self.t_acc, self.accumulation = tbuf(16 * n, cedecrt.FLOAT4, n, zero=True)
        self.t_vis, self.visibility = tbuf(16 * n, cedecrt.VISIBILITY, n, zero=True)
        # reproject="surfaces": last frame's Visibility, kept for one more frame (the two buffers swap at each frame)
        self.t_vis_prev, self.visibility_prev = tbuf(16 * n, cedecrt.VISIBILITY, n, zero=True) if self.surfaces else (None, None)
        self.t_r0, self.reservoir0 = tbuf(76 * n, cedecrt.RESERVOIR, n, zero=True, shared=True)
        self.t_r1, self.reservoir1 = tbuf(76 * n, cedecrt.RESERVOIR, n, zero=True, shared=True)
        self.t_tmp, self.temporal = tbuf(76 * n, cedecrt.RESERVOIR, n, zero=True, shared=True)
        self.bufs = self.rt.restir_buffers(self.pixels, self.accumulation, self.visibility, self.reservoir0,
                                           self.reservoir1, self.temporal)
        self.host_pixels = torch.empty(4 * W * (self.y1 - self.y0), dtype=torch.uint8).pin_memory()
        self.frame_index = 0
        self.t_cls = None
        self.halo_bytes = 0
        # pipelined read-back (download_pixels_async): copy stream, two pinned host images, the last copy's event
        self._copy_stream = None
        self._copy_events = [None, None]
        self._host_ring = None
        self._copies = 0
        self._copy_pending = None
        # ... and two device images written alternately, so that a frame's tone mapping never waits for the previous frame's copy
        self._pix_ring = None
        self._pix_cur = 0
        self._pix_copied = [None, None]
        if self.p2p and connect:
            everyone = [None] * self.world
            self.dist.all_gather_object(everyone, self.export_links())
            self.connect_links(everyone)
            self.dist.barrier()  # nobody starts rendering before every rank has opened its neighbours' buffers

    _LINKED = ("temporal", "reservoir0", "reservoir1", "scratch", "flags")

    def export_links(self):
        """what a neighbouring slab needs to store into this one: cudaIpc handles of the three reservoir buffers, the
        scratch allocation (pixel-class plane) and the flag buffer, plus the raw pointers for a neighbour that lives in
        the same process"""
        import os

        rt = self.rt
        scratch = rt.restir_reserve(self.W, self.H)
        self._flags = rt.buffer("u1", 32).zero()  # two neighbour slots + the wait kernel's time-out mark
        rt.sync()
        ptrs = {"temporal": self.temporal.ptr, "reservoir0": self.reservoir0.ptr, "reservoir1": self.reservoir1.ptr,
                "scratch": scratch, "flags": self._flags.ptr}
        return {"pid": os.getpid(), "ptr": ptrs, "ipc": {k: rt.ipc_export(v) for k, v in ptrs.items()}}

    def connect_links(self, everyone):
        """everyone[slab] = that slab's export_links(); opens the adjacent slabs' buffers and registers them"""
        import ctypes as C
        import os

        rt, n = self.rt, self.W * self.H
        links = self.c.SlabLinks()
        links.my_flags = self._flags.ptr
        self._opened = []
        for side, peer in (("up", self.rank - 1), ("down", self.rank + 1)):
            if peer < 0 or peer >= self.world:
                continue
            h = everyone[peer]
            local = h["pid"] == os.getpid()  # a handle cannot be opened by the process that exported it
            at = {k: (h["ptr"][k] if local else rt.ipc_open(h["ipc"][k])) for k in self._LINKED}
            if not local:
                self._opened += list(at.values())
            ptrs = [at["temporal"], at["reservoir0"], at["reservoir1"], at["scratch"] + 24 * n]
            getattr(links, side)[:] = (C.c_void_p * 4)(*ptrs)
            # I am the peer's "down" neighbour if it is above me, so I raise its slot 1; and vice versa
            setattr(links, side + "_flag", at["flags"] + (8 if side == "up" else 0))
        rt.slab_set_links(links)
        self._linked = True

    def close(self):
        """unlink from the neighbours and unmap their buffers (crt_ipc_close) before this slab's own buffers can go:
        a peer that still had them mapped would otherwise keep storing into freed memory.  Collective in spirit —
        every rank closes before any rank frees (callers put a barrier between close() and dropping the object)."""
        if getattr(self, "_linked", False):
            self.rt.sync()
            self.rt.slab_set_links(None)
            for p in self._opened:
                self.rt.ipc_close(p)
            self._opened = []
            self._linked = False

    def set_edges(self, edges):
        """move the slab boundaries (before any frame whose history matters: see calibrate)"""
        self.edges = list(edges)
        self.y0, self.y1 = self.edges[self.rank], self.edges[self.rank + 1]
        self.plan = halo_plan(self.H, self.edges, self.rank, self.halo) if self.world > 1 else []
        self.full_plan = full_plan(self.H, self.edges, self.rank) if self.world > 1 else []
        self.rt.set_row_range(self.y0, self.y1)
        self.host_pixels = self.torch.empty(4 * self.W * max(self.y1 - self.y0, 1), dtype=self.torch.uint8).pin_memory()

    def reset_history(self):
        self.rt.frame_join()
        with self.torch.cuda.stream(self.stream):
            for t in (self.t_tmp, self.t_r0, self.t_r1, self.t_acc):
                t.zero_()
        self.frame_index = 0

    # -- the interface bench.py uses on a SlabRenderer and on a SlabGroup alike
    slabs = property(lambda self: [self])

    def join(self):
        """order the slab's stream after everything of its frames (the overlapped tail included)"""
        self.rt.frame_join()

    def check(self):
        stage = self.rt.slab_status() if self.p2p else 0
        if stage:
            raise RuntimeError("slab %d: wait for a neighbour timed out at exchange %d" % (self.rank, stage))

    def launch_count(self):
        return self.rt.launch_count()

    def shadow_rays_traced(self):
        return self.rt.shadow_rays_traced()

    def rays_decided_at_emission(self):
        return self.rt.rays_decided_at_emission()

    def set_math_mode(self, mode):
        self.rt.set_math_mode(mode)

    def set_light_sampling(self, mode, log2_slots=0):
        self.rt.set_light_sampling(mode, log2_slots)

    def set_light_tiles(self, log2_tiles, log2_tile_size):
        self.rt.set_light_tiles(log2_tiles, log2_tile_size)

    def set_reuse_weights(self, mode):
        self.rt.set_reuse_weights(mode)

    def last_copy_events(self, slot):
        return [self._copy_events[slot]]

    def calibrate(self, rounds=2, frames=2):
        """Load balancing for a static camera: render a few throw-away frames, measure every slab's own kernel time
        (waiting for neighbours excluded), move the boundaries so that the times even out, repeat; then clear the
        history so that the real sequence starts at frame 1 with the final partition.  Returns the edges."""
        if self.world == 1:
            return self.edges
        torch, dist = self.torch, self.dist
        for _ in range(rounds):
            self.reset_history()
            self.frame()  # first frame has no temporal history: not representative
            self.rt.profile_begin()
            for _ in range(frames):
                self.frame()
            marks = self.rt.profile_end()
            mine = sum(ms for name, ms in marks if name != "signal_wait") / frames
            t = torch.zeros(self.world, dtype=torch.float64, device="cuda")
            t[self.rank] = mine
            dist.all_reduce(t)
            new_edges = rebalance(self.edges, [float(x) for x in t.tolist()], 8, HALO + 9 if self.p2p else 8)
            self.set_edges(new_edges)
        self.reset_history()
        torch.cuda.synchronize()
        dist.barrier()
        return self.edges

    def _rows(self, t, elem, a, b):
        return t[(self.H - b) * self.W * elem:(self.H - a) * self.W * elem]

    def exchange(self, t, layout):
        if self.world > 1:
            self.halo_bytes += exchange(self.dist, t, self.W, self.H, layout, self.plan)

    def set_camera(self, eye, lookat_pt):
        """a new camera for the frames that follow; with reproject=True the camera of the last frame rendered is what the
        next frame's history look-up inverts (cedecrt.RestirDI.set_camera, one slab)"""
        import numpy as np

        self.eye = tuple(float(np.float32(v)) for v in eye)
        self.raygen = self.c.lookat(eye, lookat_pt, self.W, self.H)
        self.rt.clear(self.accumulation, self.W, self.H)  # 10_restir_di.cpp:257-267

    def set_triangles(self, tris):
        """new vertices for the same triangles, in the same order (the same ones emitting): the scene array is rewritten and
        the tree refitted.  With reproject the outgoing array is kept on the device and the next frame's look-ups and, under
        unbiased weights, the history's surfaces follow the motion (crt_restir_set_previous_triangles in fused mode,
        crt_temporal_resampling_reprojected_motion in drop-in mode).  Slabs sharing this one's scene (share=) see the new
        vertices too; their frames must not be in flight (SlabGroup.set_triangles)."""
        import numpy as np

        tris = np.ascontiguousarray(tris)
        if len(tris) != self.n_tris or tris.dtype.itemsize != self.c.TRIANGLE.itemsize:
            raise ValueError("set_triangles takes the same number of triangles (%d), in the same layout" % self.n_tris)
        src = self.torch.from_numpy(tris.view(np.uint8).reshape(-1))
        self.rt.frame_join()  # the frame tail in flight may still read the vertices
        with self.torch.cuda.stream(self.stream):
            if self.reproject and not self.moved:
                if self.t_tris_prev is None:
                    self.t_tris_prev = self.torch.empty_like(self.t_tris)
                    self.prev_triangles = self.rt.wrap(self.t_tris_prev.data_ptr(), self.c.TRIANGLE, self.n_tris)
                self.t_tris_prev.copy_(self.t_tris)
                self.moved = True
            self.t_tris.copy_(src)
        self.geom.refit()  # on the context's stream, which is self.stream: after the copies

    def gather_history(self):
        """every rank's rows of the temporal reservoirs to every rank (reprojection reads the history anywhere)"""
        if self.world > 1:
            self.halo_bytes += exchange(self.dist, self.t_tmp, self.W, self.H, SOA_RESERVOIR if self.fused else AOS_RESERVOIR,
                                        self.full_plan)

    def gather_previous_visibility(self):
        """every rank's rows of last frame's Visibility to every rank (reproject="surfaces" reads it at the history pixel)"""
        if self.world > 1:
            self.halo_bytes += exchange(self.dist, self.t_vis_prev, self.W, self.H, AOS_VISIBILITY, self.full_plan)

    def _swap_visibility(self):
        """reproject="surfaces": this frame traces into the buffer two frames old; last frame's becomes the previous one"""
        self.t_vis, self.t_vis_prev = self.t_vis_prev, self.t_vis
        self.visibility, self.visibility_prev = self.visibility_prev, self.visibility
        rb = self.rt.restir_buffers
        self.bufs = rb(self.pixels, self.accumulation, self.visibility, self.reservoir0, self.reservoir1, self.temporal)
        if self._pix_ring is not None:
            self._pix_ring = [(tp, p, rb(p, self.accumulation, self.visibility, self.reservoir0, self.reservoir1, self.temporal))
                              for tp, p, _ in self._pix_ring]
            self.bufs = self._pix_ring[self._pix_cur][2]

    def frame(self):
        if self.surfaces:
            self._swap_visibility()
        rt, W, H, o, g, t, v, eye = self.rt, self.W, self.H, self.options, self.geom, self.triangles, self.visibility, self.eye
        if self.fused and self.p2p:
            for stage in range(self.n_stages()):
                self.frame_stage(stage)
            return
        self.frame_index += 1
        f = self.frame_index
        look_up = self.reproject and self.prev_raygen is not None and o.use_temporal_resampling
        motion = look_up and self.moved  # set_triangles since the last frame
        self.moved = False
        this_raygen = self.raygen
        if look_up:
            self.gather_history()
            if self.surfaces:
                self.gather_previous_visibility()
        if self.fused:
            if self.surfaces:
                rt.restir_set_previous_frame(self.prev_raygen if look_up else None, self.visibility_prev)
                self.prev_raygen = this_raygen
            elif self.reproject:
                rt.restir_set_previous_camera(self.prev_raygen if look_up else None)
                self.prev_raygen = this_raygen
            if self.reproject:
                rt.restir_set_previous_triangles(self.prev_triangles if motion else None)
            rt.restir_frame_begin(W, H, f, g, t, self.raygen, eye, self.lights, o, self.bufs)
            if self.overlap:
                rt.restir_prefetch_raycast(W, H, g, self.raygen)  # the next frame's camera (static here)
            for k in range(o.spatial_resampling_passes):  # temporal -> r1 -> r0 -> r1 (include/cedecrt.h)
                self.exchange(self.t_tmp if k == 0 else (self.t_r1 if k % 2 else self.t_r0), SOA_RESERVOIR)
                rt.restir_spatial_pass(W, H, f, k, g, t, eye, o, self.bufs)
            self._before_pixels_rewrite()
            rt.restir_frame_end(W, H, g, t, eye, o, self.bufs)
            return
        rt.raycast(W, H, g, t, self.raygen, v)
        self.exchange(self.t_vis, AOS_VISIBILITY)
        rt.generate_candidate(W, H, f, g, t, v, eye, self.lights, o, self.reservoir0)
        if motion:
            rt.temporal_resampling_reprojected_motion(W, H, f, g, t, v, eye, o, self.prev_raygen, self.prev_triangles,
                                                      self.visibility_prev if self.surfaces else None, self.temporal,
                                                      self.reservoir0)
        elif look_up and self.surfaces:
            rt.temporal_resampling_reprojected_surfaces(W, H, f, g, t, v, eye, o, self.prev_raygen, self.visibility_prev,
                                                        self.temporal, self.reservoir0)
        elif look_up:
            rt.temporal_resampling_reprojected(W, H, f, g, t, v, eye, o, self.prev_raygen, self.temporal, self.reservoir0)
        else:
            rt.temporal_resampling(W, H, f, g, t, v, eye, o, self.temporal, self.reservoir0)
        self.prev_raygen = this_raygen
        rt.save_temporal_reservoir(W, H, self.reservoir0, self.temporal)
        bi, bo, ti = self.reservoir0, self.reservoir1, self.t_r0
        for k in range(o.spatial_resampling_passes):
            if k != 0:
                bi, bo = bo, bi
                ti = self.t_r1 if ti is self.t_r0 else self.t_r0
            self.exchange(ti, AOS_RESERVOIR)
            rt.spatial_resampling(W, H, f, k, g, t, v, eye, o, bi, bo)
        rt.resolve(self.accumulation, W, H, g, t, v, eye, o, bo)
        self._before_pixels_rewrite()
        rt.tone_mapping(self.pixels, self.accumulation, W, H)

    def n_stages(self):
        return 2 + self.options.spatial_resampling_passes

    def frame_stage(self, stage):
        """the fused frame with direct halo stores, one stage per call (0: raycast + candidates + temporal; 1..passes:
        wait for the neighbours' halo rows, then one spatial pass; last: resolve + tone mapping) so that a SlabGroup can
        issue the stages of its slabs alternately"""
        rt, W, H, o, g, t, eye = self.rt, self.W, self.H, self.options, self.geom, self.triangles, self.eye
        passes = o.spatial_resampling_passes
        if stage == 0:
            self.frame_index += 1
            rt.restir_frame_begin(W, H, self.frame_index, g, t, self.raygen, eye, self.lights, o, self.bufs)
            if self.overlap:
                rt.restir_prefetch_raycast(W, H, g, self.raygen)  # the next frame's camera (static here)
        elif stage <= passes:
            k = stage - 1  # input of pass k: temporal, reservoir1, reservoir0, ...
            rt.slab_exchange(W, H, 0 if k == 0 else (2 if k % 2 else 1), self.bufs)  # rows were mirrored by the kernels
            rt.restir_spatial_pass(W, H, self.frame_index, k, g, t, eye, o, self.bufs)
        else:
            self._before_pixels_rewrite()
            rt.restir_frame_end(W, H, g, t, eye, o, self.bufs)

    def download_pixels(self):
        """the reference's read-back (10_restir_di.cpp:386-389): copy on the frame's own stream; the caller synchronises"""
        src = self._rows(self.t_pix, 4, self.y0, self.y1)
        self.rt.frame_join()
        with self.torch.cuda.stream(self.stream):
            self.host_pixels.copy_(src, non_blocking=True)

    def download_pixels_async(self):
        """Pipelined read-back: this frame's RGBA8 rows travel to pinned host memory on a copy stream while the next
        frame renders; the next frame's tone mapping (the only writer of the pixel buffer) waits for the copy.  Returns
        the index of the host image (0/1) the rows land in; wait_download(i) blocks until they are there."""
        torch = self.torch
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
        n = 4 * self.W * max(self.y1 - self.y0, 1)
        if self._host_ring is None or self._host_ring[0].numel() != n:
            self._host_ring = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(2)]
        if self._pix_ring is None:
            # the second device image; the frames from now on alternate between the two (_before_pixels_rewrite)
            import numpy as np
            npx = self.W * self.H
            t2 = torch.empty(4 * npx, dtype=torch.uint8, device=self.t_pix.device)
            p2 = self.rt.wrap(t2.data_ptr(), np.uint8, 4 * npx)
            b2 = self.rt.restir_buffers(p2, self.accumulation, self.visibility, self.reservoir0, self.reservoir1, self.temporal)
            self._pix_ring = [(self.t_pix, self.pixels, self.bufs), (t2, p2, b2)]
            self._pix_cur = 0
        slot = self._copies % 2
        self._copies += 1
        rendered = torch.cuda.Event()
        rendered.record(self._tail if self.overlap else self.stream)  # the stream tone mapping ran on
        self._copy_stream.wait_event(rendered)
        src = self._rows(self.t_pix, 4, self.y0, self.y1)
        with torch.cuda.stream(self._copy_stream):
            self._host_ring[slot].copy_(src, non_blocking=True)
            done = torch.cuda.Event()
            done.record()
        self._copy_events[slot] = done
        self._copy_pending = done
        self._pix_copied[self._pix_cur] = done
        return slot

    def wait_download(self, slot):
        if self._copy_events[slot] is not None:
            self._copy_events[slot].synchronize()
        return self._host_ring[slot]

    def _before_pixels_rewrite(self):
        """called before the kernels that write the RGBA8 image are issued.  Without pipelined read-back: nothing to order.
        With it (download_pixels_async has been called): the frame goes to the other of two device images, and only the
        copy that read that image — two frames ago — has to be over; a slow host link then delays nothing (measured on a
        box whose 33 MB copy took 5.5 ms: 12.25 ms per frame end to end with one image, the frame waiting for the
        previous copy, against 11.17 ms device-timed)."""
        if self._pix_ring is None:
            if self._copy_pending is not None:
                self.stream.wait_event(self._copy_pending)
                self._copy_pending = None
            return
        self._pix_cur ^= 1
        self.t_pix, self.pixels, self.bufs = self._pix_ring[self._pix_cur]
        ev = self._pix_copied[self._pix_cur]
        if ev is not None:
            self.stream.wait_event(ev)
            self._pix_copied[self._pix_cur] = None
        self._copy_pending = None


class SlabGroup:
    """Several row slabs per GPU, each with its own context and CUDA stream, driven by one process.

    A slab's kernels at 4 or 8 GPUs last tens to hundreds of microseconds: ten dependent launches per frame, each with
    its ramp-up and — the persistent ray tracers above all — its drain, during which most of the GPU idles.  Two
    independent kernel sequences on two streams fill each other's gaps: measured on one B200 with two slab-sized frames,
    1.29 x the throughput of one stream at 272 rows, 1.12 x at 544, 1.03 x at 2160 (profiles/overlap_probe.py).  So every
    rank renders `sub` slabs instead of one.  Slabs of one process are linked by plain device pointers, slabs of
    different processes through cudaIpc as before; scene, light list and BVH are shared by the slabs of a GPU.  The
    image is the same bit for bit (tests/gpu_slab_worker.py).

    The interface is the part of SlabRenderer's that bench.py and the tests use."""

    def __init__(self, torch, dist, rank, world, tris, cam, W, H, sub=2, options=None, overlap=False):
        self.torch, self.dist, self.rank, self.world, self.W, self.H, self.sub = torch, dist, rank, world, W, H, sub
        vworld = world * sub
        edges = [slab_rows(H, vworld, r)[0] for r in range(vworld)] + [H]
        self.stream = torch.cuda.current_stream()
        self.streams = [self.stream] + [torch.cuda.Stream() for _ in range(sub - 1)]
        self.slabs = []
        for j, st in enumerate(self.streams):
            with torch.cuda.stream(st):
                self.slabs.append(SlabRenderer(torch, dist, rank * sub + j, vworld, tris, cam, W, H, fused=True,
                                               edges=edges, options=options, p2p=True, stream=st,
                                               share=self.slabs[0] if j else None, connect=False, overlap=overlap))
        assert all(s.p2p for s in self.slabs), "slabs too thin for direct halo stores (needs >= %d rows each)" % HALO
        # One whole frame of the first slab alone, in both arithmetic modes, before any slab can wait for another: it
        # builds the shared geometry's light records and has every kernel of the frame loaded (with lazy module loading
        # a first launch waits for the device to go idle, which it never would under a spinning wait kernel).
        first = self.slabs[0]
        for mode in (first.c.MATH_FAST, first.c.MATH_LIBDEVICE, first.c.MATH_REFERENCE):
            first.rt.set_math_mode(mode)
            first.rt.restir_di_frame(W, H, 1, first.geom, first.triangles, first.raygen, first.eye, first.lights,
                                     first.options, first.bufs)
        torch.cuda.synchronize()
        mine = [s.export_links() for s in self.slabs]
        everyone = [mine]
        if world > 1:
            everyone = [None] * world
            dist.all_gather_object(everyone, mine)
        flat = [h for per_rank in everyone for h in per_rank]
        for s in self.slabs:
            s.connect_links(flat)
        self._barrier()
        self.reset_history()
        self._barrier()
        first = self.slabs[0]
        self.rt, self.geom, self.n_tris, self.n_lights, self.p2p = first.rt, first.geom, first.n_tris, first.n_lights, True
        self.halo_bytes = 0

    # -- plumbing
    def _barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    @property
    def edges(self):
        return self.slabs[0].edges

    @property
    def y0(self):
        return self.slabs[0].y0

    @property
    def y1(self):
        return self.slabs[-1].y1

    def check(self):
        """raise if a slab's wait for a neighbour timed out (csrc/slab_p2p.cu: k_signal_wait)"""
        for s in self.slabs:
            stage = s.rt.slab_status()
            if stage:
                raise RuntimeError("slab %d: wait for a neighbour timed out at exchange %d" % (s.rank, stage))

    def join(self):
        """the group's first stream (the one callers time and synchronise) waits for the other slabs' streams"""
        for s in self.slabs:
            s.join()
        for st in self.streams[1:]:
            ev = self.torch.cuda.Event()
            ev.record(st)
            self.stream.wait_event(ev)

    def fork(self):
        """the other slabs' streams wait for what has been issued to the first one"""
        ev = self.torch.cuda.Event()
        ev.record(self.stream)
        for st in self.streams[1:]:
            st.wait_event(ev)

    def frame(self):
        # stage by stage over the slabs, so that every stream always has the next kernel queued
        for stage in range(self.slabs[0].n_stages()):
            for s in self.slabs:
                s.frame_stage(stage)
        # a wait that gave up (4 s watchdog of k_signal_wait) means stale halo rows: never render on silently.  The
        # status read synchronises the stream, so it is taken every 64th frame only.
        self._frames = getattr(self, "_frames", 0) + 1
        if self._frames % 64 == 0:
            self.check()

    def close(self):
        for s in self.slabs:
            s.close()

    def reset_history(self):
        for s in self.slabs:
            s.reset_history()

    def set_camera(self, eye, lookat_pt):
        for s in self.slabs:
            s.set_camera(eye, lookat_pt)

    def set_triangles(self, tris):
        """new vertices for the same triangles: the slabs of this GPU share one scene array and one tree, so every slab's
        frame is finished first and the first slab rewrites the array and refits.  The slabs run over direct-store links,
        which refuse reprojection, so there is no previous array to pass on (as RestirDI(reproject=False))."""
        self._barrier()
        self.slabs[0].set_triangles(tris)
        self._barrier()

    def set_edges(self, edges):
        for s in self.slabs:
            s.set_edges(edges)

    def calibrate(self, rounds=3, frames=4):
        """as SlabRenderer.calibrate, over all slabs of all ranks; a slab's time is measured while the GPU is shared with
        the rank's other slabs, which is the condition it will run under"""
        torch = self.torch
        vworld = self.world * self.sub
        for _ in range(rounds):
            self._barrier()
            self.reset_history()
            self._barrier()
            self.frame()
            for s in self.slabs:
                s.rt.profile_begin()
            for _ in range(frames):
                self.frame()
            t = torch.zeros(vworld, dtype=torch.float64, device="cuda")
            for s in self.slabs:
                marks = s.rt.profile_end()
                t[s.rank] = sum(ms for name, ms in marks if name != "signal_wait") / frames
            if self.world > 1:
                self.dist.all_reduce(t)
            self.set_edges(rebalance(self.edges, [float(x) for x in t.tolist()], 8, HALO + 9))
        self._barrier()
        self.reset_history()
        self._barrier()
        return self.edges

    # -- what bench.py reads
    def launch_count(self):
        return sum(s.rt.launch_count() for s in self.slabs)

    def shadow_rays_traced(self):
        a = [s.rt.shadow_rays_traced() for s in self.slabs]
        return sum(x[0] for x in a), sum(x[1] for x in a)

    def rays_decided_at_emission(self):
        a = [s.rt.rays_decided_at_emission() for s in self.slabs]
        return sum(x[0] for x in a), sum(x[1] for x in a)

    def set_math_mode(self, mode):
        for s in self.slabs:
            s.rt.set_math_mode(mode)

    def set_light_sampling(self, mode, log2_slots=0):
        for s in self.slabs:
            s.rt.set_light_sampling(mode, log2_slots)

    def set_light_tiles(self, log2_tiles, log2_tile_size):
        for s in self.slabs:
            s.rt.set_light_tiles(log2_tiles, log2_tile_size)

    def set_reuse_weights(self, mode):
        for s in self.slabs:
            s.rt.set_reuse_weights(mode)

    def download_pixels(self):
        for s in self.slabs:
            s.download_pixels()

    def download_pixels_async(self):
        return [s.download_pixels_async() for s in self.slabs]

    def wait_download(self, slots):
        return [s.wait_download(k) for s, k in zip(self.slabs, slots)]

    def last_copy_events(self, slots):
        return [s._copy_events[k] for s, k in zip(self.slabs, slots)]

    def _rows(self, t, elem, a, b):
        return self.slabs[0]._rows(t, elem, a, b)
