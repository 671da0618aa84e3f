"""Multi-GPU support: environment-batch sharding and the (only) collective, an off-path statistics reduction.

Environments are independent, so ``parallel_envs`` shards across GPUs with no communication on the step path
(SURVEY.md section 8e): one process per GPU, each with its own buffers and CUDA graph.  Randomness is keyed by the
GLOBAL environment index (``env_offset`` + local index), so a shard draws the same random numbers as its slice of the
whole batch.  Its trajectories equal that slice's as long as the reference's two batch-wide conditions agree between
the shard and the whole batch: "every environment is terminated / truncated" (utils/env.py:212) and "this agent has no
task in any environment" (wildfire.py:434, rideshare.py:276).  Each shard evaluates them over its own environments, so
when they differ (one shard entirely terminated, an agent with tasks only in another shard) the shard behaves like the
reference run on that shard alone.  The statistics record is reduced with one ``all_reduce`` (NCCL over NVLink on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.distributed as dist


def shard(total_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous block of environments owned by ``rank``: returns (env_offset, parallel_envs)."""
    if not 0 <= rank < world_size:
        raise ValueError(f'rank {rank} outside [0, {world_size})')
    base, extra = divmod(total_envs, world_size)
    count = base + (1 if rank < extra else 0)
    offset = rank * base + min(rank, extra)
    return offset, count


def episode_statistics(cumulative_rewards: torch.Tensor, terminated: torch.Tensor, truncated: torch.Tensor,
                       num_moves: torch.Tensor) -> torch.Tensor:
    """float64 record [3 + A]: env-steps executed, #terminated, #truncated, sum of cumulative reward per agent."""
    head = torch.stack([num_moves.sum().double(), terminated.sum().double(), truncated.sum().double()])
    return torch.cat([head, cumulative_rewards.double().sum(dim=0)])


def all_reduce_statistics(record: torch.Tensor, group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """Sum the statistics record over every rank (no-op without an initialised process group)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(record, op=dist.ReduceOp.SUM, group=group)
    return record
