"""Episode statistics of every rollout route against the route's own output streams.

Every kernel that steps envs also keeps the per-env step counter and running return and folds finished episodes into
the statistics stripes (cx_episode.cuh).  Here each route's full stats() dict must equal what its own reward and flag
streams imply, recomputed on the host: an episode ends on a TERMINATED or TRUNCATED step that counts (neither
BAD_ACTION nor ALREADY_OVER), its return is the float32 running sum of the rewards of its counted steps (as the kernels
keep it), its length the number of those steps.  Rewards of these worlds are small integers, so the float64 sums are
exact in any order, and all routes agree with each other as a consequence."""
import numpy as np
import pytest
import torch

from campx_b200 import _native as N
from examples.generality_worlds import make_generality_world
from examples.worlds import make_world

pytestmark = pytest.mark.gpu

T, LIMIT = 40, 13              # every env truncates at least once; with auto_reset=False it is frozen afterwards
ALIGNED, RAGGED = 4128, 4099   # 4,128 = 129 warps of 32 but not a whole number of 64-env tiles: the rest goes to the
                               # lane kernel; 4,099 runs the scalar / ragged paths

# how a route is driven: CX_ROUTE for cx_rollout, T single steps, or a call of its own
AGENT_ROUTES = ["auto", "tile64", "tile128", "tile256", "lane", "obs", "step_composer", "no_step_composer",
                "rollout_observations", "rollout_policy"]
GENERIC_ROUTES = ["auto", "gen96", "gen80", "gen_wave"]
# rollout_policy picks its own actions for whole warps of 32 envs: aligned batch only
CASES = [(w, r, n) for w, routes in (("goal", AGENT_ROUTES), ("hello", GENERIC_ROUTES), ("goal2", GENERIC_ROUTES))
         for r in routes for n in (ALIGNED, RAGGED) if not (r == "rollout_policy" and n % 32)]


def _engine(world, n, auto_reset):
    kw = dict(num_envs=n, max_episode_steps=LIMIT, track_returns=True, auto_reset=auto_reset, verify=False)
    game = make_world(world, **kw) if world == "hello" else make_generality_world(world, **kw)
    game.its_showtime()
    return game


def _run(g, route, monkeypatch):
    """T steps of every env through `route` -> (reward, flags) [T, n]"""
    n = g.num_envs
    if route in ("auto", "rollout_observations", "rollout_policy"):
        monkeypatch.delenv("CX_ROUTE", raising=False)
    else:
        monkeypatch.setenv("CX_ROUTE", route)
    if route == "rollout_policy":   # the kernel samples its own actions
        gen = torch.Generator(device="cuda").manual_seed(3)
        feat, hidden = g.n_chars * g.cells, 32
        # small weights: nearly uniform actions, so that episodes end at the exit, in the pit and at the time limit
        w1t = 0.1 * torch.randn((feat, hidden), generator=gen, device="cuda")
        b1 = 0.1 * torch.randn(hidden, generator=gen, device="cuda")
        w2 = 0.1 * torch.randn((g.n_actions, hidden), generator=gen, device="cuda")
        b2 = 0.1 * torch.randn(g.n_actions, generator=gen, device="cuda")
        states = torch.empty((T + 1, n, feat), dtype=torch.float32, device="cuda")
        actions = torch.empty((T, n), dtype=torch.uint8, device="cuda")
        reward = torch.empty((T, n), dtype=torch.float32, device="cuda")
        flags = torch.empty((T, n), dtype=torch.uint8, device="cuda")
        g.rollout_policy(T, w1t, b1, w2, b2, 11, states, actions, reward, flags)
        assert len(torch.unique(actions)) > 1
        return reward, flags
    acts = g.fill_actions(T, seed=5)
    acts[3, ::7] = 9                                                   # a few actions outside the action set
    board, reward, flags, disc = g.alloc_outputs(T)
    if route in ("step_composer", "no_step_composer"):
        for t in range(T):
            g.step(acts[t].contiguous(), board[t], reward[t], flags[t], None if disc is None else disc[t])
    elif route == "rollout_observations":
        layered = torch.empty((T, n, g.n_chars, g.rows, g.cols), dtype=torch.uint8, device="cuda")
        g.rollout_observations(acts, board, layered, reward, flags, disc)
    else:
        g.rollout(acts, board, reward, flags, disc)
    return reward, flags


def _implied_stats(reward, flags):
    """stats() of envs that start a fresh episode, implied by their [T, n] reward and flag streams"""
    r, f = reward.cpu().numpy(), flags.cpu().numpy()
    n = r.shape[1]
    ret = np.zeros(n, dtype=np.float32)
    length = np.zeros(n, dtype=np.int64)
    returns, lengths = [], []
    for t in range(r.shape[0]):
        counts = (f[t] & (N.CX_FLAG_BAD_ACTION | N.CX_FLAG_ALREADY_OVER)) == 0
        ret = np.where(counts, ret + r[t], ret)                        # float32, as the kernels keep it
        length += counts
        ended = counts & ((f[t] & (N.CX_FLAG_TERMINATED | N.CX_FLAG_TRUNCATED)) != 0)
        returns.append(ret[ended].astype(np.float64))
        lengths.append(length[ended])
        ret[ended] = 0.0
        length[ended] = 0
    ret_all, len_all = np.concatenate(returns), np.concatenate(lengths)
    return {"episodes": float(len(ret_all)), "return_sum": float(ret_all.sum()),
            "return_sumsq": float((ret_all * ret_all).sum()), "length_sum": float(len_all.sum()),
            "return_max": float(ret_all.max()), "neg_return_min": float((-ret_all).max()),
            "env_steps": float(r.size), "reserved": 0.0}


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("world,route,n", CASES)
def test_stats_are_what_the_streams_imply(world, route, n, auto_reset, monkeypatch):
    game = _engine(world, n, auto_reset)
    g = game.native
    reward, flags = _run(g, route, monkeypatch)
    want = _implied_stats(reward, flags)
    assert want["episodes"] > 0
    if not auto_reset:   # every env ended once by the time limit and was frozen from then on
        assert int(((flags & N.CX_FLAG_ALREADY_OVER) != 0).sum()) > 0
    assert g.stats() == want
