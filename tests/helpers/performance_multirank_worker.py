"""Worker of tests/test_gpu_performance.py::test_two_ranks_reduce_to_one_gpu, launched by torchrun with one rank per GPU.

Rank r steps envs [r*n, (r+1)*n) of a global boat_race batch that tracks the safety performance (Philox actions keyed
by the global env id); the episode statistics go through all_reduce_stats and rank 0 compares them, performance_sum
included, with one single-GPU run of the whole batch.  Prints PERFORMANCE_MULTIRANK_OK on success.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import torch
import torch.distributed as dist

from campx_b200 import _native as N
from campx_b200 import dist as cxdist
from examples.worlds import BOAT_RACE_REGIONS, make_world


def _run(n, env_offset, T=40, seed=543):
    game = make_world("boat_race", num_envs=n, max_episode_steps=16, track_returns=True, verify=False,
                      performance_regions=BOAT_RACE_REGIONS)
    game.its_showtime()
    game.rollout_random(T, seed, env_offset=env_offset)
    return game.native.stats_tensor.clone()


def main():
    n = int(sys.argv[1])
    rank, world, local_rank = cxdist.init_from_env()
    torch.cuda.set_device(local_rank)
    stats = _run(n, rank * n)
    cxdist.all_reduce_stats(stats)
    if rank == 0:
        one = _run(world * n, 0)
        assert one[N.CX_STAT_PERFORMANCE_SUM] != 0.0
        assert torch.equal(stats, one), (stats.tolist(), one.tolist())
        print("PERFORMANCE_MULTIRANK_OK world=%d envs_per_rank=%d" % (world, n), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
