"""Scene sharding across the GPUs of one box.  Scenes are independent (offline_main.py:32-34: every scene owns
its TrackBuffer and ring), so the hot loop needs no collective; the only exchange is the gather of the packed
per-scene results (mmw_pack_results) at the end of a run or every K frames."""
from __future__ import annotations

from typing import List, Tuple


def shard_bounds(n_scenes: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous block [lo, hi) of global scene ids owned by ``rank``; blocks differ by at most one scene."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError("bad world/rank")
    base, rem = divmod(n_scenes, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_scene_ids(n_scenes: int, world: int, rank: int) -> List[int]:
    lo, hi = shard_bounds(n_scenes, world, rank)
    return list(range(lo, hi))


def gather_results(local, n_scenes: int, per_scene: int, group=None):
    """All-gathers the packed per-scene result rows of every rank into global scene order.
    ``local``: torch tensor [local_scenes * per_scene] (CUDA with nccl, CPU with gloo).  Ranks may own a
    different number of scenes, so shards are padded to the largest one for the collective."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    sizes = [shard_bounds(n_scenes, world, r) for r in range(world)]
    max_local = max(hi - lo for lo, hi in sizes)
    pad = torch.zeros(max_local * per_scene, dtype=local.dtype, device=local.device)
    pad[:local.numel()] = local
    out = torch.empty(world * max_local * per_scene, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, pad, group=group)
    parts = [out[r * max_local * per_scene: r * max_local * per_scene + (hi - lo) * per_scene]
             for r, (lo, hi) in enumerate(sizes)]
    return torch.cat(parts)


def move_scenes(src, src_scenes, dst, dst_scenes=None, reset_source=True):
    """Moves live scenes from BatchedTracker ``src`` to ``dst`` (e.g. to drain a GPU or rebalance ranks): exports
    ``src_scenes``, imports them into ``dst_scenes`` (default: the same indices) with their tracks, rings, id counters
    and sensor-table entries, then, with ``reset_source``, frees the source slots (``src.reset_scenes``).  The contexts
    must have the same max_points, max_tracks and frames_batch; they may sit on different GPUs.  Returns the blob."""
    import numpy as np
    src_idx = np.ascontiguousarray(np.atleast_1d(src_scenes), dtype=np.int32).reshape(-1)
    dst_idx = src_idx if dst_scenes is None else np.ascontiguousarray(np.atleast_1d(dst_scenes), dtype=np.int32).reshape(-1)
    if dst_idx.size != src_idx.size:
        raise ValueError("move_scenes: %d source scenes but %d destination slots" % (src_idx.size, dst_idx.size))
    if reset_source and src is dst and np.intersect1d(src_idx, dst_idx).size:
        raise ValueError("move_scenes: resetting the source would clear scenes just moved into the same context")
    blob = src.export_scenes(src_idx)
    dst.import_scenes(blob, dst_idx)
    if reset_source:
        src.reset_scenes(src_idx)
    return blob


class NcclGather:
    """The result gather through the C ABI (mmw_gather_nccl): one ncclAllGather on the context's stream, this rank's
    records packed straight into its block of the output.  The communicator is formed with the library's own helpers;
    the 128-byte id travels over the already initialised torch.distributed group (any backend)."""

    def __init__(self, tracker, group=None):
        import ctypes as C
        import numpy as np
        import torch
        import torch.distributed as dist
        from . import _lib
        self.bt, self.lib = tracker, tracker.lib
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        ident = np.zeros(128, np.uint8)
        if self.rank == 0:
            _lib.check(self.lib.mmw_nccl_unique_id(_lib.ptr(ident)))
        box = [ident.tobytes()]
        dist.broadcast_object_list(box, src=0, group=group)
        ident = np.frombuffer(box[0], np.uint8).copy()
        comm = C.c_void_p()
        _lib.check(self.lib.mmw_nccl_comm_init(tracker._h, _lib.ptr(ident), self.world, self.rank, C.byref(comm)))
        self.comm = comm
        self.out = torch.empty(self.world * tracker.S * tracker.tcap * _lib.RESULT_FLOATS, dtype=torch.float32,
                               device=torch.device("cuda", tracker.device))

    def gather(self):
        """All ranks' packed records, [world * S * max_tracks * 72] fp32 on this rank's device (after sync())."""
        from . import _lib
        import ctypes as C
        _lib.check(self.lib.mmw_gather_nccl(self.bt._h, self.comm, self.world, C.c_void_p(self.out.data_ptr())))
        return self.out

    def close(self):
        from . import _lib
        if self.comm:
            _lib.check(self.lib.mmw_nccl_comm_destroy(self.comm))
            self.comm = None
