"""Multi-GPU sharding of the environment axis (SURVEY §8e).

Environments are independent, so GPU g of G owns the contiguous env range
[g*N/G, (g+1)*N/G) with its own copy of the track tables, its own state arrays and its own
slice of the action stream; the step and GAE kernels need NO collective.  Only rollout
statistics (train.py:272-274, avg_reward) cross the shards: one small all-reduce.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist


def shard_range(n_total: int, world_size: int, rank: int) -> tuple[int, int]:
    """Contiguous, balanced partition: the first (n_total % world_size) ranks own one extra env."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, extra = divmod(n_total, world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def track_blocks(n_total: int, n_tracks: int, lo: int, hi: int) -> np.ndarray:
    """Track of each global env lo .. hi - 1 when n_total envs share n_tracks tracks: env g runs on track
    g * n_tracks // n_total, i.e. contiguous, balanced blocks (warps of the fused rollout kernel are then nearly all
    single-track), independent of how the envs are sharded.  int32 [hi - lo]."""
    if not (1 <= n_tracks <= n_total):
        raise ValueError("need 1 <= n_tracks <= n_total")
    if not (0 <= lo <= hi <= n_total):
        raise ValueError("env range out of bounds")
    return (np.arange(lo, hi, dtype=np.int64) * n_tracks // n_total).astype(np.int32)


def allreduce_rollout_stats(reward_sum: torch.Tensor, n_steps: torch.Tensor, episodes: torch.Tensor | None = None):
    """Sum (reward_sum, n_steps[, episodes]) over all ranks; returns python floats.
    avg_reward of train.py:272 = reward_sum / n_steps after the reduction."""
    parts = [reward_sum.reshape(1).double(), n_steps.reshape(1).double()]
    if episodes is not None:
        parts.append(episodes.reshape(1).double())
    buf = torch.cat(parts)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
    return tuple(float(x) for x in buf.tolist())
