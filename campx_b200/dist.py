"""Multi-GPU plumbing: one process per GPU, environments sharded by rank, NO collective on the step
path (environments are independent: SURVEY section 8(e)).  The only exchange is the all-reduce of the
8-double episode-statistics block, issued per reporting interval over NCCL (NVLink 5 / NVSwitch); the
same code runs over gloo on CPU tensors for tests.
"""
import os

import torch
import torch.distributed as dist

from . import _native as N

SUM_SLOTS = [0, 1, 2, 3, 6, 7]  # episodes, return_sum, return_sumsq, length_sum, env_steps, performance_sum (0
                                # for games that do not track performance)
MAX_SLOTS = [4, 5]              # return_max, -return_min


def init_from_env(backend=None):
    """Initialise torch.distributed from torchrun's environment; returns (rank, world, local_rank)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        kwargs = {}
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
            kwargs["device_id"] = torch.device("cuda", local_rank)
        dist.init_process_group(backend=backend, rank=rank, world_size=world, **kwargs)
    return rank, world, local_rank


def shard_range(n_total, rank, world):
    """Contiguous block of environments owned by `rank` (remainder spread over the first ranks)."""
    base, rem = divmod(int(n_total), int(world))
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def all_reduce_stats(stats, group=None):
    """In-place all-reduce of a float64[8] episode-statistics block (CX_STAT_* layout).

    Two collectives of 40 and 16 bytes: SUM over the additive slots, MAX over (max, -min).
    Returns the reduced tensor; a no-op without an initialised process group.
    """
    if stats.dtype != torch.float64 or stats.numel() != N.CX_STATS_DOUBLES:
        raise ValueError("stats must be float64[%d]" % N.CX_STATS_DOUBLES)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return stats
    sums = stats[SUM_SLOTS].contiguous()
    maxs = stats[MAX_SLOTS].contiguous()
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(maxs, op=dist.ReduceOp.MAX, group=group)
    stats[SUM_SLOTS] = sums
    stats[MAX_SLOTS] = maxs
    return stats


def summarize_stats(stats, performance=False):
    """float64[8] block -> dict with mean/std/min/max episode return and mean length; with `performance`, also the
    mean safety performance of the episodes (games created with performance_regions)."""
    s = [float(v) for v in stats.tolist()]
    n = s[0]
    out = {"episodes": n, "env_steps": s[6]}
    if n > 0:
        mean = s[1] / n
        out.update(return_mean=mean, return_std=max(s[2] / n - mean * mean, 0.0) ** 0.5,
                   return_max=s[4], return_min=-s[5], length_mean=s[3] / n)
        if performance:
            out["performance_mean"] = s[N.CX_STAT_PERFORMANCE_SUM] / n
    return out
