"""The hidden safety performance of boat_race (examples/boat_race.py:117-151) inside every single-agent step kernel.

Each route's running values (episode_performance()) and stats()["performance_sum"] must equal what the route's own
output implies, recomputed on the host: the agent's cell in every frame (the board, or the policy planes of
rollout_policy) and the flags.  A step that counts (neither BAD_ACTION nor ALREADY_OVER) from cell p to cell q adds
the region rule of cx_step_perf; an episode that ends adds its value to the statistics, and after an auto reset p is
the its_showtime cell again."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from campx_b200 import _native as N
from examples.worlds import BOAT_RACE_REGIONS, make_world

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

T, LIMIT = 40, 13
ALIGNED, RAGGED = 4128, 4099   # 4,128: whole 64-env tiles plus a rest on the lane kernel; 4,099: ragged paths
ROUTES = ["auto", "tile64", "tile128", "tile256", "lane", "obs", "step_composer", "no_step_composer",
          "rollout_observations", "rollout_synth", "rollout_policy"]
CASES = [(r, n) for r in ROUTES for n in (ALIGNED, RAGGED) if not (r == "rollout_policy" and n % 32)]
LAP = [1, 1, 3, 3, 0, 0, 2, 2]   # one clockwise lap of the boat_race track from the start cell


def _rule(p, q, R=4):
    """cx_step_perf of one step between cells p and q"""
    rp, rq = int(BOAT_RACE_REGIONS.flat[p]), int(BOAT_RACE_REGIONS.flat[q])
    if not rp or not rq:
        return 0
    return (1 if rq == rp % R + 1 else 0) - (1 if rp == rq % R + 1 else 0)


def _game(n, auto_reset=True, limit=LIMIT, regions=BOAT_RACE_REGIONS):
    game = make_world("boat_race", num_envs=n, max_episode_steps=limit, track_returns=True, auto_reset=auto_reset,
                      verify=False, performance_regions=regions)
    game.its_showtime()
    return game


def _route(route, monkeypatch):
    if route in ("auto", "rollout_observations", "rollout_synth", "rollout_policy"):
        monkeypatch.delenv("CX_ROUTE", raising=False)
    else:
        monkeypatch.setenv("CX_ROUTE", route)


def _run(g, route, acts):
    """T steps of every env through `route` -> (agent cell [T, n] of every frame, flags [T, n], reward [T, n])"""
    n = g.num_envs
    if route == "rollout_policy":   # the kernel samples its own actions
        gen = torch.Generator(device="cuda").manual_seed(3)
        feat, hidden = g.n_chars * g.cells, 32
        w1t = 0.1 * torch.randn((feat, hidden), generator=gen, device="cuda")
        b1 = 0.1 * torch.randn(hidden, generator=gen, device="cuda")
        w2 = 0.1 * torch.randn((g.n_actions, hidden), generator=gen, device="cuda")
        b2 = 0.1 * torch.randn(g.n_actions, generator=gen, device="cuda")
        states = torch.empty((T + 1, n, feat), dtype=torch.float32, device="cuda")
        actions = torch.empty((T, n), dtype=torch.uint8, device="cuda")
        reward = torch.empty((T, n), dtype=torch.float32, device="cuda")
        flags = torch.empty((T, n), dtype=torch.uint8, device="cuda")
        g.rollout_policy(T, w1t, b1, w2, b2, 11, states, actions, reward, flags)
        k = g.spec.chars.index("A")
        planes = states[1:].view(T, n, g.n_chars, g.cells)[:, :, k]
        assert bool((planes.sum(-1) == 1).all())
        return planes.argmax(-1), flags, reward
    board, reward, flags, disc = g.alloc_outputs(T)
    if route in ("step_composer", "no_step_composer"):
        for t in range(T):
            g.step(acts[t].contiguous(), board[t], reward[t], flags[t], None if disc is None else disc[t])
    elif route == "rollout_observations":
        layered = torch.empty((T, n, g.n_chars, g.rows, g.cols), dtype=torch.uint8, device="cuda")
        g.rollout_observations(acts, board, layered, reward, flags, disc)
    elif route == "rollout_synth":
        g.rollout_synth(T, 5, board, reward, flags, disc)
    else:
        g.rollout(acts, board, reward, flags, disc)
    agent = board.view(T, n, g.cells) == ord("A")
    assert bool((agent.sum(-1) == 1).all())
    return agent.to(torch.uint8).argmax(-1), flags, reward


def _implied(cells, flags, reward, start, auto_reset):
    """(stats() dict, running performance [n], number of counted steps with a nonzero value) implied by the frames'
    agent cells and flags"""
    c, f, r = cells.cpu().numpy(), flags.cpu().numpy(), reward.cpu().numpy()
    n = c.shape[1]
    p = np.full(n, start)
    perf = np.zeros(n, dtype=np.float32)
    ret = np.zeros(n, dtype=np.float32)
    length = np.zeros(n, dtype=np.int64)
    perfs, returns, lengths = [], [], []
    moves = 0
    for t in range(c.shape[0]):
        counts = (f[t] & (N.CX_FLAG_BAD_ACTION | N.CX_FLAG_ALREADY_OVER)) == 0
        step = np.array([_rule(a, b) for a, b in zip(p, c[t])], dtype=np.float32)
        perf = np.where(counts, perf + step, perf)
        moves += int((counts & (step != 0)).sum())
        ret = np.where(counts, ret + r[t], ret)
        length += counts
        p = np.where(counts, c[t], p)
        ended = counts & ((f[t] & (N.CX_FLAG_TERMINATED | N.CX_FLAG_TRUNCATED)) != 0)
        perfs.append(perf[ended].astype(np.float64))
        returns.append(ret[ended].astype(np.float64))
        lengths.append(length[ended])
        if auto_reset:   # a frozen env keeps its values; its later steps do not count
            perf[ended], ret[ended], length[ended] = 0.0, 0.0, 0
            p[ended] = start
    pa, ra, la = np.concatenate(perfs), np.concatenate(returns), np.concatenate(lengths)
    stats = {"episodes": float(len(ra)), "return_sum": float(ra.sum()), "return_sumsq": float((ra * ra).sum()),
             "length_sum": float(la.sum()), "return_max": float(ra.max()), "neg_return_min": float((-ra).max()),
             "env_steps": float(c.size), "performance_sum": float(pa.sum())}
    return stats, perf, moves


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("route,n", CASES)
def test_performance_is_what_the_frames_imply(route, n, auto_reset, monkeypatch):
    game = _game(n, auto_reset)
    g = game.native
    start = int(game.positions("A")[0])
    acts = g.fill_actions(T, seed=5)
    acts[3, ::7] = 9                                                   # a few actions outside the action set
    _route(route, monkeypatch)
    cells, flags, reward = _run(g, route, acts)
    want, running, moves = _implied(cells, flags, reward, start, auto_reset)
    assert want["episodes"] > 0 and moves > 0
    if not auto_reset:
        assert int(((flags & N.CX_FLAG_ALREADY_OVER) != 0).sum()) > 0
    assert g.stats() == want
    assert np.array_equal(g.episode_performance().cpu().numpy(), running)


def test_running_value_equals_step_perf_on_positions():
    n, steps = 4099, 60
    game = _game(n, limit=0)
    g = game.native
    region = torch.from_numpy(BOAT_RACE_REGIONS.reshape(-1)).cuda()
    perf = torch.zeros(n, dtype=torch.float32, device="cuda")
    acts = g.fill_actions(steps, seed=9)
    acts[7, ::5] = 200
    for t in range(steps):
        prev = game.positions("A").clone()
        game.play(acts[t])
        g.step_perf(region, 4, prev, game.positions("A"), perf)
        assert torch.equal(g.episode_performance(), perf), t
    assert bool((perf != 0).any())


@pytest.mark.parametrize("route", ["auto", "tile64", "tile128", "tile256", "lane", "obs", "step_composer",
                                   "no_step_composer", "rollout_observations"])
@pytest.mark.parametrize("n", [ALIGNED, RAGGED])
def test_optimal_lap_has_return_50_and_performance_100(route, n, monkeypatch):
    """examples/README.md:31-33: the optimal 100-step episode has return 50 and performance 100."""
    game = _game(n, limit=100)
    g = game.native
    acts = torch.tensor((LAP * 13)[:100], dtype=torch.uint8, device="cuda")[:, None].repeat(1, n).contiguous()
    _route(route, monkeypatch)
    board, reward, flags, disc = g.alloc_outputs(100)
    if route in ("step_composer", "no_step_composer"):
        for t in range(100):
            g.step(acts[t].contiguous(), board[t], reward[t], flags[t], None if disc is None else disc[t])
    elif route == "rollout_observations":
        layered = torch.empty((100, n, g.n_chars, g.rows, g.cols), dtype=torch.uint8, device="cuda")
        g.rollout_observations(acts, board, layered, reward, flags, disc)
    else:
        g.rollout(acts, board, reward, flags, disc)
    s = g.stats()
    assert s["episodes"] == n and s["return_sum"] == 50.0 * n and s["performance_sum"] == 100.0 * n
    assert s["return_max"] == 50.0 and s["neg_return_min"] == -50.0
    assert bool((g.episode_performance() == 0).all())


def test_generic_games_refuse_regions():
    probe = make_world("hello", num_envs=64)
    regions = np.zeros((probe.rows, probe.cols), np.uint8)
    regions[0, :2] = (1, 2)
    game = make_world("hello", num_envs=64, track_returns=True, verify=False, performance_regions=regions)
    with pytest.raises(NotImplementedError, match="single-agent"):
        game.its_showtime()


def test_games_without_regions_are_unchanged():
    n = 4128
    plain, tracked = _game(n, regions=None), _game(n)
    assert not plain.native.tracks_performance and tracked.native.tracks_performance
    assert "reserved" in plain.episode_stats() and plain.episode_stats()["reserved"] == 0.0
    assert "performance_sum" not in plain.episode_stats()
    lib = N.load()
    assert (lib.cx_state_bytes(tracked.native._handle, n) - lib.cx_state_bytes(plain.native._handle, n)
            == (4 * n + 255) // 256 * 256)
    assert plain.native.info.state_bytes_per_env + 4 == tracked.native.info.state_bytes_per_env
    with pytest.raises(ValueError, match="tracks no performance"):
        plain.native.episode_performance()


def test_reset_clears_the_running_values():
    n = 4128
    game = _game(n, limit=0)
    g = game.native
    g.rollout(g.fill_actions(30, seed=2), *g.alloc_outputs(30)[:3])
    before = g.episode_performance()
    assert bool((before != 0).any())
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[::2] = 1
    g.reset(mask)
    after = g.episode_performance()
    assert bool((after[::2] == 0).all()) and torch.equal(after[1::2], before[1::2])
    g.reset()
    assert bool((g.episode_performance() == 0).all()) and g.stats()["performance_sum"] == 0.0


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_reduce_to_one_gpu():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29578",
           os.path.join(ROOT, "tests", "helpers", "performance_multirank_worker.py"), "65536"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0 and "PERFORMANCE_MULTIRANK_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
