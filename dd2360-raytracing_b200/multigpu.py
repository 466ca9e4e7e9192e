"""Frame sharding over ranks (one process per GPU, torch.distributed for the plumbing).

The reference is single-GPU.  A frame partitions naturally (SURVEY §8e):
  * tiles : rank g renders the interleaved 8x4 pixel tiles {g, g+G, g+2G, ...} with ALL ns samples and the unmodified
            per-pixel stream, zeros elsewhere.  The sum over ranks is bit-identical to the 1-GPU frame.
  * spp   : rank g renders ns/G samples of every pixel from streams seeded 1984 + pixel_index + g*num_pixels.
            Statistically equivalent, not bit-identical (per-pixel samples are chained through the RNG, D8).
Either way the partial LINEAR radiance buffers are combined with ONE collective over NCCL/NVLink — a reduce-scatter:
rank r receives the summed elements [r*S, (r+1)*S) of the flattened frame, applies /ns and sqrt (main.cu:111-114) to
its own slice and, for a host destination, copies that slice into a pinned host frame that all ranks of the box map
(POSIX shared memory registered with cudaHostRegister) — N PCIe links work in parallel and no rank funnels the
whole frame.  `reduce_frame` (sum onto one rank) is kept for callers that want the frame on one GPU.

Stream order: the library launches on the stream handed to RayTracer.set_stream (torch's current stream in
bench.py); torch.distributed orders its NCCL stream against that same stream, so render -> collective -> finalise ->
copy need no host synchronisation.  When the RayTracer runs on its own stream instead, `render_sharded` bridges the
two with the context's blocking stream semantics plus an explicit synchronize.
"""
from __future__ import annotations

import mmap
import os

import numpy as np

from . import PREC_FP16, PREC_FP32, SHARD_NONE, SHARD_SPP, SHARD_TILES, RayTracer

TILE_W, TILE_H = 8, 4


def tile_owner_map(nx: int, ny: int, world: int) -> np.ndarray:
    """[ny, nx] int32: which rank owns each pixel under RT_SHARD_TILES (tile index modulo world size)."""
    tx = (nx + TILE_W - 1) // TILE_W
    jj, ii = np.meshgrid(np.arange(ny), np.arange(nx), indexing="ij")
    tile = (jj // TILE_H) * tx + (ii // TILE_W)
    return (tile % world).astype(np.int32)


def spp_share(ns: int, rank: int, world: int) -> int:
    """Samples per pixel rank `rank` traces under RT_SHARD_SPP."""
    return ns // world + (1 if rank < ns % world else 0)


def slice_elems(total: int, world: int) -> int:
    """Elements per rank of the reduce-scatter: the flattened frame padded up to a multiple of the world size."""
    return (total + world - 1) // world


def slice_range(total: int, rank: int, world: int) -> tuple[int, int]:
    """[begin, end) of the REAL frame elements rank `rank` owns after the reduce-scatter (the last slice may be short)."""
    s = slice_elems(total, world)
    return min(rank * s, total), min((rank + 1) * s, total)


def reduce_frame(accum, dist, dst: int = 0):
    """Sum the ranks' linear radiance buffers onto `dst` (in place)."""
    if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
        dist.reduce(accum, dst=dst, op=dist.ReduceOp.SUM)
    return accum


def reduce_scatter_frame(accum_padded, out_slice, dist):
    """The one collective of the path: out_slice = sum over ranks of accum_padded[rank*S : (rank+1)*S]."""
    if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
        dist.reduce_scatter_tensor(out_slice, accum_padded, op=dist.ReduceOp.SUM)
    else:
        out_slice.copy_(accum_padded[: out_slice.numel()])
    return out_slice


class SharedHostFrame:
    """A host frame every rank of the box can write its slice into: POSIX shared memory, page-locked in each process
    (cudaHostRegister) so that device->host copies run at PCIe speed and asynchronously.  Rank 0 creates it."""

    def __init__(self, name: str, nbytes: int, create: bool, torch):
        self.name, self.nbytes, self.torch = name, nbytes, torch
        path = os.path.join("/dev/shm", name)
        flags = os.O_RDWR | (os.O_CREAT if create else 0)
        fd = os.open(path, flags, 0o600)
        try:
            if create:
                os.ftruncate(fd, nbytes)
            self.map = mmap.mmap(fd, nbytes)
        finally:
            os.close(fd)
        self.path, self.owner = path, create
        self.array = np.frombuffer(self.map, dtype=np.float32)
        self.tensor = torch.from_numpy(self.array)
        self.registered = False
        if torch.cuda.is_available():
            rc = torch.cuda.cudart().cudaHostRegister(self.tensor.data_ptr(), nbytes, 0)
            self.registered = int(rc) == 0

    def close(self):
        if self.registered:
            self.torch.cuda.cudart().cudaHostUnregister(self.tensor.data_ptr())
            self.registered = False
        self.tensor = None
        self.array = None
        try:
            self.map.close()
        except BufferError:
            pass
        if self.owner and os.path.exists(self.path):
            os.unlink(self.path)


class ShardedFrame:
    """Per-rank buffers of a sharded frame: the padded linear accumulator, this rank's slice, optionally the shared host frame."""

    def __init__(self, torch, device, nx: int, ny: int, rank: int, world: int):
        self.torch, self.nx, self.ny, self.rank, self.world = torch, nx, ny, rank, world
        self.total = nx * ny * 3
        self.S = slice_elems(self.total, world)
        self.accum = torch.zeros(self.S * world, dtype=torch.float32, device=device)   # the pad stays 0
        self.slice = torch.empty(self.S, dtype=torch.float32, device=device)
        self.begin, self.end = slice_range(self.total, rank, world)
        self.host = None

    def attach_host(self, host: SharedHostFrame):
        self.host = host

    def frame_view(self):
        return self.accum[: self.total].view(self.ny, self.nx, 3)


def render_sharded(rt: RayTracer, frame: ShardedFrame, ns: int, use_octree: bool, mode: int = SHARD_TILES, dist=None,
                   want_stats: bool = True, to_host: bool = False, precision: int = PREC_FP32):
    """Render this rank's shard, reduce-scatter the linear sums, finalise this rank's slice (and copy it to the shared host
    frame when `to_host`).  Everything is queued on the RayTracer's stream / torch's current stream; the caller
    synchronises.  Returns the per-rank render stats (None without want_stats).  PREC_FP16 frames shard by tiles only:
    spp shards would each hold the half sum of ns/G samples, a different image from the 1-GPU one."""
    if precision == PREC_FP16 and mode == SHARD_SPP:
        raise ValueError("USE_FP16 frames shard by tiles only (SHARD_TILES): spp shards' half sums do not add up to the 1-GPU frame")
    world, rank = frame.world, frame.rank
    args = rt.args(frame.nx, frame.ny, ns, use_octree, shard_mode=mode if world > 1 else SHARD_NONE, shard_rank=rank, shard_count=world,
                   precision=precision)
    # the render is queued WITHOUT waiting for its statistics, so that the collective, the finalise kernel and the copy are
    # queued right behind it (no host round trip in the middle of the frame); the statistics are read at the end
    world_sharded = world > 1
    st = rt.render_accumulate(args, frame.accum.data_ptr(), want_stats=want_stats and not world_sharded)
    reduce_scatter_frame(frame.accum, frame.slice, dist)
    rt.finalize_ex(frame.slice.data_ptr(), frame.slice.data_ptr(), frame.S, ns, precision)
    if to_host and frame.host is not None and frame.end > frame.begin:
        frame.host.tensor[frame.begin:frame.end].copy_(frame.slice[: frame.end - frame.begin], non_blocking=True)
    if want_stats and world_sharded:
        st = rt.last_render_stats()
    return st


__all__ = ["tile_owner_map", "spp_share", "slice_elems", "slice_range", "reduce_frame", "reduce_scatter_frame", "SharedHostFrame",
           "ShardedFrame", "render_sharded", "SHARD_TILES", "SHARD_SPP", "SHARD_NONE"]
