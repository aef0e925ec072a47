"""Development aid: k_agent_rollout (256 envs per warp) against the lane-per-env kernel by batch size: run it under
CX_ROUTE=tile256 and CX_ROUTE=obs."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from scripts.quick_time import run
for n in [int(a) for a in sys.argv[1:]] or (16384, 65536, 262144):
    run("demo1", n, 32, 30, max_episode_steps=100, track_returns=True)
