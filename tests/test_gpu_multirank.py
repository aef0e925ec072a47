"""One process per GPU under torchrun (NCCL): an N-rank run reproduces ONE single-GPU run of the whole batch, env for
env (SURVEY 8(e)).  Needs >= 2 visible GPUs; on a one-GPU box the single-process form of the same property is
tests/test_gpu_engine.py::test_rollout_equals_play_and_sharding_is_deterministic."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("n", [4096, 600000])      # lane-per-env kernel; k_agent_rollout (tile builds)
def test_n_ranks_reproduce_one_gpu_env_for_env(n):
    world = min(torch.cuda.device_count(), 8)
    if n > 100000:
        world = min(world, 2)                       # the single-GPU twin holds world * n envs of Hello World boards
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", "29577",
           os.path.join(ROOT, "tests", "helpers", "multirank_worker.py"), str(n)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0 and "MULTIRANK_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
