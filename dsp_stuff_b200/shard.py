"""Channel sharding across ranks (SURVEY.md section 8e): every channel owns its state, shared parameters are
replicated and per-channel ones (Engine.set_f32_channels) are sliced: rank r's engine gets values[lo:hi] with
(lo, hi) = channel_range(r, ...).  Per-channel impulse responses (Engine.set_taps_channels) pass the whole bank with
set_index[lo:hi].  So the path partitions with no data-path collective.  The only collective is the optional gather of
output blocks to rank 0.  The FFT FIR pairs channels of one impulse response inside aligned groups of 32 channels, so a
shard whose lo is a multiple of 32 reproduces the whole run bit for bit; other boundaries agree within rounding."""
from __future__ import annotations

from typing import Optional, Tuple


def channel_range(rank: int, world: int, total_channels: int) -> Tuple[int, int]:
    """Contiguous, balanced ranges: rank r owns [lo, hi).  The first (total % world) ranks get one extra."""
    if not (0 <= rank < world) or total_channels < 0:
        raise ValueError("bad rank/world/total")
    base, extra = divmod(total_channels, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def gather_to_rank0(local, total_channels: int, group=None):
    """Gathers each rank's [C_r x n] output block to rank 0 (NCCL on GPUs, gloo on CPU).  Returns the
    [total_channels x n] tensor on rank 0 and None elsewhere.  Uneven shards are padded to the largest."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    sizes = [channel_range(r, world, total_channels) for r in range(world)]
    cmax = max(hi - lo for lo, hi in sizes)
    n = local.shape[1]
    padded = local
    if local.shape[0] != cmax:
        padded = torch.zeros((cmax, n), dtype=local.dtype, device=local.device)
        padded[: local.shape[0]] = local
    bufs = [torch.empty_like(padded) for _ in range(world)] if rank == 0 else None
    dist.gather(padded.contiguous(), bufs, dst=0, group=group)
    if rank != 0:
        return None
    return torch.cat([bufs[r][: hi - lo] for r, (lo, hi) in enumerate(sizes)], dim=0)
