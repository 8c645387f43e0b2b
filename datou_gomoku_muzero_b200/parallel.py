"""Multi-GPU plumbing: one process per GPU, games sharded across ranks, no collective on the
per-simulation path (SURVEY section 8e).  torch.distributed (NCCL on GPUs, gloo in CPU tests) is used
only for the two exchanges the reference does through multiprocessing queues:

  * trainer -> workers weight publication (`model_update_queue`, workers.py:587-593, 331-335)
    -> `broadcast_weights`: one flattened-buffer broadcast from the trainer rank;
  * workers -> data loader trajectories (`data_queue`, workers.py:230, 399)
    -> `gather_packed_games`: counts all-gathered, fixed-stride move records gathered as raw bytes.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist


def shard_games(total_games: int, world_size: int, rank: int):
    """Contiguous shard [start, stop) of the global game indices owned by `rank` (sizes differ by <= 1)."""
    base, extra = divmod(int(total_games), int(world_size))
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def rank_noise_seed(base_seed: int, rank: int) -> int:
    """Distinct Gumbel-noise stream per rank (games on different GPUs must not share noise)."""
    return (int(base_seed) * 0x9E3779B1 + 0x85EBCA6B * (rank + 1)) & 0x7FFFFFFFFFFFFFFF


def broadcast_weights(module: torch.nn.Module, src: int = 0, group=None):
    """Publish `module`'s parameters and buffers from `src` to every rank with ONE broadcast of a flat
    buffer per dtype (88 MB fp32 at 15x15: launch latency matters, link count does not)."""
    tensors = [t for t in list(module.parameters()) + list(module.buffers())]
    by_dtype = {}
    for t in tensors:
        by_dtype.setdefault(t.dtype, []).append(t)
    for dtype, ts in by_dtype.items():
        flat = torch.cat([t.detach().reshape(-1) for t in ts])
        dist.broadcast(flat, src=src, group=group)
        off = 0
        for t in ts:
            n = t.numel()
            with torch.no_grad():
                t.copy_(flat[off:off + n].reshape(t.shape))
            off += n
    return module


class FlatWeights:
    """A module's parameters and buffers re-homed as views into ONE flat tensor per dtype, so that publishing
    the weights (`model_update_queue`, workers.py:587-593) is a single in-place broadcast per dtype with no
    packing or unpacking kernels -- the link, not ~300 small copies, sets the time.  The module keeps working
    as before (its tensors now alias the flat buffers); every rank must wrap an identically shaped module."""

    def __init__(self, module: torch.nn.Module):
        self.module = module
        groups = {}
        for t in list(module.parameters()) + list(module.buffers()):
            groups.setdefault((t.dtype, t.device), []).append(t)
        self.flats = []
        for (dtype, device), ts in groups.items():
            flat = torch.empty(sum(t.numel() for t in ts), dtype=dtype, device=device)
            off = 0
            for t in ts:
                n = t.numel()
                view = flat[off:off + n].view(t.shape)
                with torch.no_grad():
                    view.copy_(t)
                t.data = view                     # parameter / buffer now aliases the flat storage
                off += n
            self.flats.append(flat)

    @property
    def nbytes(self):
        return sum(f.numel() * f.element_size() for f in self.flats)

    def broadcast(self, src: int = 0, group=None):
        for f in self.flats:
            dist.broadcast(f, src=src, group=group)
        return self.module


def max_over_ranks(value: float, device=None, group=None) -> float:
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())


def sum_over_ranks(value: float, device=None, group=None) -> float:
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return float(t.item())


def gather_packed_games(packed, board_size, dst: int = 0, group=None, device=None):
    """The reference's `data_queue` (workers.py:230, 399) across ranks: every rank's finished games, as packed move
    records (trajectory.PackedGames, fixed stride ~4.7 KB per move at 15x15), gathered on rank `dst` with tensor
    collectives -- `all_gather` of the (moves, games) counts, then one `gather` of the record bytes and one of the
    game tables, each padded to the largest rank.  No pickling, no per-game Python objects; with NCCL the records go
    GPU -> GPU.  `packed` may be None (this rank has nothing).  Returns a PackedGames on `dst` whose table has a
    fifth column = source rank; None elsewhere."""
    from .trajectory import PackedGames, record_dtype
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    stride = record_dtype(board_size).itemsize
    if device is None:
        device = packed.records.device if packed is not None and torch.is_tensor(packed.records) else torch.device("cpu")
    m = 0 if packed is None else packed.n_moves
    n = 0 if packed is None else len(packed)
    mine = torch.tensor([m, n], dtype=torch.int64, device=device)
    counts = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(counts, mine, group=group)
    counts = torch.stack(counts).cpu().numpy()
    M, Nn = int(counts[:, 0].max()), int(counts[:, 1].max())
    if M == 0:
        return None
    rec = torch.zeros((M, stride), dtype=torch.uint8, device=device)
    tab = torch.zeros((Nn, 4), dtype=torch.int32, device=device)
    if m:
        rec[:m].copy_(torch.as_tensor(packed.records).reshape(m, stride))
        tab[:n].copy_(torch.as_tensor(np.ascontiguousarray(packed.table[:, :4], dtype=np.int32)))
    recs = [torch.empty_like(rec) for _ in range(world)] if rank == dst else None
    tabs = [torch.empty_like(tab) for _ in range(world)] if rank == dst else None
    dist.gather(rec, recs, dst=dst, group=group)
    dist.gather(tab, tabs, dst=dst, group=group)
    if rank != dst:
        return None
    out_rec = torch.cat([recs[r][:counts[r, 0]] for r in range(world)])
    tables, offs, base = [], [0], 0
    for r in range(world):
        t = tabs[r][:counts[r, 1]].cpu().numpy()
        tables.append(np.concatenate([t, np.full((len(t), 1), r, np.int32)], axis=1))
        for L in t[:, 2]:
            base += int(L); offs.append(base)
    return PackedGames(out_rec, np.concatenate(tables), np.asarray(offs, np.int64), board_size)


def gather_finished_games(records, dst: int = 0, group=None):
    """Harvested games as Python dicts (TrajectoryStore.harvest) of every rank -> `dst`, through
    `gather_object` (pickle).  Convenience for small jobs and tests; the tensor path is gather_packed_games."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    counts = [None] * world
    dist.all_gather_object(counts, len(records), group=group)
    gathered = [None] * world if rank == dst else None
    dist.gather_object(records, gathered, dst=dst, group=group)
    if rank != dst:
        return None
    out = []
    for r, recs in enumerate(gathered):
        assert len(recs) == counts[r]
        for rec in recs:
            rec = dict(rec)
            rec["rank"] = r
            out.append(rec)
    return out
