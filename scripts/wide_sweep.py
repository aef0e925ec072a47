"""Development aid: single-agent worlds of several board sizes by batch size and kernel route (CX_ROUTE: lane =
k_agent_rollout_lane, obs = lane-per-env TMA kernel, tile64 = k_agent_rollout; boards above 96 cells run on the obs
kernel under tile64 as well)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from campx_b200 import things
from campx_b200.ascii_art import ascii_art_to_game, Partial
from campx_b200.runtime import NativeGame
from examples.worlds import Walker
from tests.test_gpu_generic_worlds import _random_art

def run(rows, cols, n, T, route):
    os.environ["CX_ROUTE"] = route
    art = _random_art(np.random.Generator(np.random.PCG64(rows * cols)), rows, cols, 0.2, 0.2)
    game = ascii_art_to_game(art, ' ', drapes={'A': Partial(Walker, walls='#', treasures='*'),
                                               '#': things.FixedDrape, '*': things.FixedDrape},
                             z_order='*A#', num_envs=n, max_episode_steps=100, track_returns=True, verify=False)
    g = NativeGame(game.compile(), n)
    nb = max(2, int(500e6 // (n * T * (g.cells + 6))) + 1)
    bufs = [g.alloc_outputs(T) for _ in range(nb)]
    acts = [g.fill_actions(T, seed=543, t0=i * T) for i in range(nb)]
    def timed(lead, count):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        for i in range(lead): g.rollout(acts[i % nb], *bufs[i % nb])
        e0.record()
        for i in range(count): g.rollout(acts[i % nb], *bufs[i % nb])
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / count
    per = timed(2, 4)
    timed(0, max(4, int(60 / per)))
    ms = timed(2, max(8, int(60 / per)))
    balg = 1 + 4 + 1 + g.cells + 14.0 / T
    print("%dx%d (%d cells) n=%d T=%d %s: %.4f ms/launch  %.0f GB/s (%.1f%%)" % (
        rows, cols, g.cells, n, T, route, ms, n * T * balg / ms / 1e6, n * T * balg / ms / 1e6 / 65.341), flush=True)

if __name__ == "__main__":
    for rows, cols in ((5, 5), (8, 12), (10, 12), (15, 16)):
        for n in (16384, 65536, 1 << 18, 1 << 20):
            for route in ("lane", "obs", "tile64"):
                run(rows, cols, n, 16, route)
