"""Multi-GPU plumbing: one process per GPU, series / chains sharded across ranks.

The path shards naturally (SURVEY.md section 8e): every series or chain is independent, so a
rank owns a contiguous block of the batch and there is NO data-path collective.  The only
inter-GPU traffic is an optional sum-reduce of per-rank scalars (log-likelihood totals, pooled
Gibbs sufficient statistics) over ``torch.distributed`` (NCCL on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

from typing import Tuple


def shard_range(total: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous block [lo, hi) of ``total`` series owned by ``rank``: sizes differ by at most
    one, earlier ranks get the larger blocks, the union over ranks is exactly [0, total)."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError(f"bad rank/world {rank}/{world}")
    base, extra = divmod(int(total), int(world))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def time_chunk(total_T: int, rank: int, world: int) -> Tuple[int, int, int]:
    """Rank's chunk of ONE series of ``total_T`` observations cut along time (the time-sharded scan):
    observations y[lo:hi] and ``first_row``, the global row of the chunk's first row.  Rank 0 also holds
    row 0, the prior (keep_init = 1), so its rows are 0 .. hi and every later rank's first row is
    1 + lo.  Every chunk holds at least one observation: world <= total_T."""
    if int(world) > int(total_T):
        raise ValueError(f"{world} ranks for {total_T} observations: every chunk needs one")
    lo, hi = shard_range(total_T, rank, world)
    return lo, hi, 0 if rank == 0 else lo + 1


def wave_aligned_slabs(lo: int, hi: int, wave: int, waves_per_launch: int):
    """Split a rank's block into launches of whole GPU waves (last one takes the remainder)."""
    per = max(1, int(wave) * max(1, int(waves_per_launch)))
    out, b = [], lo
    while b < hi:
        out.append((b, min(hi, b + per)))
        b += per
    return out


def reduce_sum(tensor):
    """In-place sum over ranks when a process group is initialised; identity otherwise."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(tensor, op=dist.ReduceOp.SUM)
    return tensor


def reduce_max(tensor):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(tensor, op=dist.ReduceOp.MAX)
    return tensor
