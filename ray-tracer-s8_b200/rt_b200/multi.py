"""Tile scheduler over the GPUs of one box.

The reference scatters row bands over slaves with HTTP and gathers `ImageSlice` callbacks
(ray-tracer-controller/src/main.rs:47-75,79-93,109-115).  Here the frame is cut into 8x4-pixel tiles,
tile t belongs to rank `tile_owner(t, ranks)` (a rotating interleave, so sky-heavy and object-heavy
regions spread evenly), the scene is replicated on every GPU like the reference replicates it in every
request body, and the frame is assembled on rank 0.  Two drivers:

  * `FrameScheduler` — one process per GPU, torch.distributed for the plumbing (setup only):
      - "p2p"  (fused render + gather): rank 0 owns the frame in its HBM and exports a CUDA IPC handle; every
        other rank maps it and its render kernel stores finished tiles straight into rank 0's memory over
        NVLink.  Each tile's completion is released into per-slab counters in the frame's control block, so
        rank 0 knows when a slab is final WITHOUT a barrier between the ranks, and copies it to the host
        while the other slabs still render.
      - "nccl" (baseline): every rank renders its tiles into a zeroed local frame; an NCCL reduce(MAX) over the
        uint8 frames to rank 0 assembles them (tiles are disjoint, everything else is zero).
  * `MultiDeviceRenderer` — ONE process drives all GPUs through the C ABI (`rt_render_frame_multi`): what a
    Rust controller / slave links against; no torch, no IPC handles.

Pixels draw from per-pixel streams, so the image does not depend on the partition.
"""
from __future__ import annotations

import numpy as np

TILE_W, TILE_H = 8, 4  # must match csrc/rt_device.cuh


def tile_grid(width: int, height: int):
    return (width + TILE_W - 1) // TILE_W, (height + TILE_H - 1) // TILE_H


def tile_owner(tile: int, ranks: int) -> int:
    """Rank that renders global tile index `tile` (row-major over the tile grid).

    Inverse of the kernel's ticket map g = k*ranks + (rank + k) % ranks  (csrc/rt_kernels.cu)."""
    k, e = divmod(tile, ranks)
    return (e - k) % ranks


def owner_map(width: int, height: int, ranks: int) -> np.ndarray:
    """int32 (height, width): owning rank of every pixel."""
    tx, ty = tile_grid(width, height)
    t = np.arange(tx * ty, dtype=np.int64)
    own = ((t % ranks) - (t // ranks)) % ranks
    own = own.reshape(ty, tx).astype(np.int32)
    return np.repeat(np.repeat(own, TILE_H, axis=0), TILE_W, axis=1)[:height, :width]


def tiles_of_rank(width: int, height: int, rank: int, ranks: int) -> np.ndarray:
    tx, ty = tile_grid(width, height)
    t = np.arange(tx * ty, dtype=np.int64)
    return t[((t % ranks) - (t // ranks)) % ranks == rank]


def assemble_reduce(frame, dst: int = 0, group=None):
    """Assemble disjoint, zero-padded per-rank frames on `dst` with reduce(MAX).  Works on any backend
    (NCCL on GPU tensors; gloo on CPU tensors in the tests)."""
    import torch.distributed as dist

    dist.reduce(frame, dst=dst, op=dist.ReduceOp.MAX, group=group)
    return frame


class FrameScheduler:
    """Per-rank driver of a multi-GPU frame.  `ctx` is this rank's rt_b200.Context.

    p2p mode keeps TWO frames on rank 0 and alternates between them, so a rank that is done with frame f may start
    frame f + 1 while rank 0 still collects f; before a rank writes into a buffer again it waits — on the device, by
    polling the buffer's control block over NVLink — until rank 0 has collected the frame that was in it."""

    N_BUFFERS = 2

    def __init__(self, ctx, rank: int, world_size: int, mode: str = "p2p"):
        self.ctx, self.rank, self.world = ctx, rank, world_size
        self.mode = mode
        self._frames = []         # device pointers (rank 0: owned; others: peer mappings)
        self._frame_bytes = 0
        self._local = None
        self._owns = False
        self.frames_done = 0      # frames rendered so far

    # -- frame buffers ---------------------------------------------------------------------------------
    def setup(self, width: int, height: int):
        nbytes = width * height * 3
        self.close()
        self._frame_bytes = nbytes
        self.frames_done = 0
        if self.world == 1:
            self._frames = [self.ctx.frame_alloc(nbytes)[0]]
            self._owns = True
            return self
        import torch
        import torch.distributed as dist

        if self.mode == "p2p":
            obj = [None]
            if self.rank == 0:
                pairs = [self.ctx.frame_alloc(nbytes) for _ in range(self.N_BUFFERS)]
                self._frames = [p for p, _ in pairs]
                self._owns = True
                obj = [[h for _, h in pairs]]
            dist.broadcast_object_list(obj, src=0)
            if self.rank != 0:
                self._frames = [self.ctx.frame_open(h) for h in obj[0]]
        elif self.mode == "nccl":
            self._local = torch.zeros(nbytes, dtype=torch.uint8, device=f"cuda:{self.ctx.device}")
            self._frames = [self._local.data_ptr()]
        else:
            raise ValueError(f"unknown mode {self.mode!r}")
        return self

    def close(self):
        if self._local is None:
            for p in self._frames:
                if self._owns:
                    self.ctx.frame_free(p)
                else:
                    self.ctx.frame_close(p)
        self._frames, self._local, self._owns = [], None, False

    @property
    def frame_ptr(self) -> int:
        """Device pointer of the frame the last render() went into."""
        return self._frames[(self.frames_done - 1) % len(self._frames)]

    # -- one frame -----------------------------------------------------------------------------------
    def render(self, scene, params, want_stats: bool = False, out: np.ndarray | None = None):
        """Render this rank's tiles; on rank 0 return when the WHOLE frame is complete (device resident, and in
        `out` — host memory, rank 0 only — when given).  Ranks do not synchronise with each other on the host: rank 0
        watches the frame's completion counters on its device."""
        f = self.frames_done
        self.frames_done += 1
        buf = self._frames[f % len(self._frames)]
        seq = f // len(self._frames) + 1          # this is the seq-th frame of that buffer
        if self.world > 1 and self.mode == "nccl":
            import torch

            self._local.zero_()
            torch.cuda.current_stream().synchronize()
            st = self.ctx.render_tiles_device(scene, params, self.rank, self.world, buf, sync=True, want_stats=True)
            assemble_reduce(self._local, 0)
            torch.cuda.current_stream().synchronize()
            if out is not None and self.rank == 0:
                self.ctx.frame_download(buf, out)
            return st if want_stats else None
        if self.rank == 0 and self.world > 1:
            # own tiles + the whole frame: into `out` slab by slab, or (out None) just complete on the device
            st = self.ctx.render_tiles_collect(scene, params, 0, self.world, buf, seq, out, want_stats=True)
        else:
            if self.rank != 0:
                self.ctx.frame_wait_consumed(buf, self._frame_bytes, seq - 1)   # device-side, before the kernel
            st = self.ctx.render_tiles_device(scene, params, self.rank, self.world, buf, sync=True, want_stats=True)
            if out is not None and self.rank == 0:
                self.ctx.frame_download(buf, out)
        return st if want_stats else None

    def download(self, out: np.ndarray) -> np.ndarray:
        """Rank 0: copy the last assembled frame to host memory."""
        assert self.rank == 0
        return self.ctx.frame_download(self.frame_ptr, out)


class MultiDeviceRenderer:
    """All GPUs of the box from one process, through `rt_render_frame_multi` (no torch, no IPC).

    `devices` = CUDA device indices; device[0] owns the frame.  One scene copy per device, like one request body per
    slave in the reference (controller main.rs:47-75)."""

    def __init__(self, devices):
        from . import api

        self._api = api
        self.ctxs = [api.Context(d) for d in devices]

    def scenes(self, spheres=None, triangles=None, world_index=None):
        return [c.scene(spheres, triangles, world_index) for c in self.ctxs]

    def render(self, scenes, params, out: np.ndarray | None = None, want_stats: bool = False):
        return self._api.render_frame_multi(self.ctxs, scenes, params, out=out, want_stats=want_stats)

    def render_jpeg(self, scenes, params, quality: int = 90, want_stats: bool = False):
        """The frame of render() as JPEG bytes, encoded on the first GPU where the frame lies (rt_render_frame_jpeg)."""
        return self._api.render_frame_jpeg(self.ctxs, scenes, params, quality=quality, want_stats=want_stats)

    def render_progressive(self, scene_per_ctx, params, schedule=(1, 1, 2, 4, 8)):
        """Preview that improves, on every GPU: yields (samples_done, frame) after each chunk of `schedule` samples; each
        frame equals render() at spp = samples_done (rt_render_samples_multi; params.divisions must be 1)."""
        accs = [c.accum(params) for c in self.ctxs]
        try:
            for n in schedule:
                frame = self._api.render_samples_multi(self.ctxs, scene_per_ctx, accs, n)
                yield accs[0].samples, frame
        finally:
            for a in accs:
                a.close()

    def close(self):
        for c in self.ctxs:
            c.close()
        self.ctxs = []
