"""Sprite agents that walls stop (PyColab's MazeWalker: CX_KIND_SPRITE with blockers) on the GPU, against the sprite
oracle (tests/helpers/sprite_oracle.py, unpinned by the reference) frame for frame: board, layers, reward, discount,
flags and the agent's cell, through every route and entry point that runs them.  A sprite agent behind a drape runs
on the single-agent kernels (info.path == 1) and is, there, the same game as its one-cell-drape twin; every other
sprite game runs on the generic kernels (info.path == 2)."""
import numpy as np
import pytest
import torch

from campx_b200 import _native as N
from campx_b200 import things
from campx_b200.ascii_art import Partial, ascii_art_to_game
from examples.generality_worlds import Drifter
from examples.worlds import BOAT_RACE_REGIONS, Runner, make_world
from tests.helpers import sprite_oracle as S

pytestmark = pytest.mark.gpu
T, LIMIT = 80, 40
ALIGNED, RAGGED, SMALL = 4128, 4099, 64
AGENT_ROUTES = ["auto", "tile64", "tile128", "tile256", "lane", "obs", "step_composer", "no_step_composer",
                "rollout_observations", "step_observations_f32", "rollout_policy", "policy_sample_board"]
GENERIC_ROUTES = ["gen96", "gen80", "gen_wave"]
LAP = [1, 1, 3, 3, 0, 0, 2, 2]   # one clockwise lap of the boat_race track from the start cell
_GAMES = {}


def world(name, n, **kw):
    """Un-started Engine of sprite_oracle world `name`, written with the user classes."""
    if name in ('maze', 'sprite_race', 'boat_race'):
        return make_world(name, num_envs=n, **kw)
    if name in ('drift', 'groups'):
        schedule = 'AS#' if name == 'drift' else [['S'], ['A', '#']]
        return ascii_art_to_game(S.DRIFT_ART, ' ', sprites={'A': Partial(Runner, walls='#', per_step=1.0), 'S': Drifter},
                                 drapes={'#': things.FixedDrape}, z_order='#SA', update_schedule=schedule,
                                 num_envs=n, **kw)
    if name == 'stamp':
        return ascii_art_to_game(S.STAMP_ART, ' ', sprites={'A': Partial(Runner, walls='#~', per_step=0.5)},
                                 drapes={'#': things.FixedDrape}, z_order='A#', update_schedule='A#', num_envs=n, **kw)
    raise KeyError(name)


def _game(name, n, auto_reset=True, limit=LIMIT, **kw):
    key = (name, n, auto_reset, limit, repr(sorted(kw.items())))
    if key not in _GAMES:
        g = world(name, n, max_episode_steps=limit, auto_reset=auto_reset, track_returns=True, **kw)
        g.its_showtime()
        _GAMES[key] = g
    g = _GAMES[key]
    g.reset()
    return g


def _route(route, monkeypatch):
    """CX_ROUTE for the kernel routes; the entry points (rollout_observations, ...) run with automatic selection"""
    if route in ("tile64", "tile128", "tile256", "lane", "obs", "step_composer", "no_step_composer") + \
            tuple(GENERIC_ROUTES):
        monkeypatch.setenv("CX_ROUTE", route)
    else:
        monkeypatch.delenv("CX_ROUTE", raising=False)


def _policy(g, hidden=32):
    gen = torch.Generator(device="cuda").manual_seed(3)
    feat = g.n_chars * g.cells
    return (0.1 * torch.randn((feat, hidden), generator=gen, device="cuda"),
            0.1 * torch.randn(hidden, generator=gen, device="cuda"),
            0.1 * torch.randn((g.n_actions, hidden), generator=gen, device="cuda"),
            0.1 * torch.randn(g.n_actions, generator=gen, device="cuda"))


def _actions(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 5, size=(T, n)).astype(np.uint8)
    a[rng.random((T, n)) < 0.02] = 9          # now and then an action outside the set
    return torch.from_numpy(a).cuda()


def _run(game, route, acts):
    """-> (actions, board or None, layered or None, reward, discount or None, flags) of T steps through `route`"""
    g, n = game.native, game.num_envs
    if route == "rollout_policy":
        w1t, b1, w2, b2 = _policy(g)
        states = torch.empty((T + 1, n, g.n_chars * g.cells), dtype=torch.float32, device="cuda")
        acts = torch.empty((T, n), dtype=torch.uint8, device="cuda")
        reward = torch.empty((T, n), dtype=torch.float32, device="cuda")
        flags = torch.empty((T, n), dtype=torch.uint8, device="cuda")
        g.rollout_policy(T, w1t, b1, w2, b2, 11, states, acts, reward, flags)
        return acts, None, states[1:].view(T, n, g.n_chars, g.rows, g.cols), reward, None, flags
    board, reward, flags, disc = g.alloc_outputs(T, discount=True)
    layered = None
    if route == "rollout_observations":
        layered = torch.empty((T, n, g.n_chars, g.rows, g.cols), dtype=torch.uint8, device="cuda")
        g.rollout_observations(acts, board, layered, reward, flags, disc)
    elif route == "step_observations_f32":
        layered = torch.empty((T, n, g.n_chars, g.rows, g.cols), dtype=torch.float32, device="cuda")
        for t in range(T):
            g.step_observations(acts[t].contiguous(), board[t], layered[t], reward[t], flags[t], disc[t])
    elif route == "policy_sample_board":
        w1t, b1, w2, b2 = _policy(g)
        acts = torch.empty((T, n), dtype=torch.uint8, device="cuda")
        prev = g.render()
        for t in range(T):
            acts[t] = g.policy_sample_board(prev, w1t, b1, w2, b2, 13, step_offset=t)
            g.step(acts[t].contiguous(), board[t], reward[t], flags[t], disc[t])
            prev = board[t]
    elif route in ("step_composer", "no_step_composer"):
        for t in range(T):
            g.step(acts[t].contiguous(), board[t], reward[t], flags[t], disc[t])
    else:
        g.rollout(acts, board, reward, flags, disc)
    return acts, board, layered, reward, disc, flags


def _envs(n):
    return sorted(i for i in {0, 1, n // 2, n - 1} | ({31, 32, 63, 4096} if n > 64 else {5, 17}) if i < n)


def _compare(name, out, auto_reset, envs, limit=LIMIT, occlusion_in_layers=True):
    acts, board, layered, reward, disc, flags = (None if x is None else x.cpu().numpy() for x in out)
    for i in envs:
        for t, (b, lay, r, d, f, _) in enumerate(S.rollout(name, acts[:, i], limit, auto_reset, occlusion_in_layers)):
            ctx = (name, i, t, int(acts[t, i]))
            if board is not None:
                assert np.array_equal(board[t, i], b), ctx
            if layered is not None:
                assert np.array_equal(layered[t, i], lay.astype(layered.dtype)), ctx
            assert float(reward[t, i]) == r and int(flags[t, i]) == f, ctx
            if disc is not None:
                assert float(disc[t, i]) == d, ctx


def _implied_stats(reward, flags):
    """stats() that the reward and flag streams imply (as tests/test_gpu_episode_stats.py)"""
    r, f = reward.cpu().numpy(), flags.cpu().numpy()
    n = r.shape[1]
    ret, steps = np.zeros(n, np.float32), np.zeros(n)
    eps = ret_sum = len_sum = 0.0
    for t in range(r.shape[0]):
        counts = (f[t] & (N.CX_FLAG_BAD_ACTION | N.CX_FLAG_ALREADY_OVER)) == 0
        ret = np.where(counts, ret + r[t], ret).astype(np.float32)
        steps += counts
        done = counts & ((f[t] & (N.CX_FLAG_TERMINATED | N.CX_FLAG_TRUNCATED)) != 0)
        eps += done.sum()
        ret_sum += ret[done].astype(np.float64).sum()
        len_sum += steps[done].sum()
        ret[done], steps[done] = 0, 0
    return eps, ret_sum, len_sum, float(r.size)


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("n", [ALIGNED, RAGGED, SMALL])
@pytest.mark.parametrize("route", AGENT_ROUTES)
@pytest.mark.parametrize("name", ["maze", "sprite_race"])
def test_agent_path_matches_the_oracle(name, route, n, auto_reset, monkeypatch):
    if route == "rollout_policy" and n % 32:
        pytest.skip("cx_rollout_policy takes multiples of 32 envs")
    game = _game(name, n, auto_reset)
    assert game.native.info.path == N.CX_PATH_AGENT
    _route(route, monkeypatch)
    out = _run(game, route, _actions(n, n + len(route)))
    _compare(name, out, auto_reset, _envs(n))
    eps, ret_sum, len_sum, steps = _implied_stats(out[3], out[5])
    s = game.native.stats()
    assert s["episodes"] == eps and s["length_sum"] == len_sum and s["env_steps"] == steps
    assert abs(s["return_sum"] - ret_sum) <= 1e-6 * max(1.0, abs(ret_sum))
    if auto_reset:
        assert eps > 0


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("n", [RAGGED, SMALL])
@pytest.mark.parametrize("route", GENERIC_ROUTES)
@pytest.mark.parametrize("name", ["drift", "stamp", "groups"])
def test_generic_path_matches_the_oracle(name, route, n, auto_reset, monkeypatch):
    game = _game(name, n, auto_reset)
    info = game.native.info
    assert info.path == N.CX_PATH_GENERIC and bool(info.has_dynamic_backdrop) == (name == "stamp")
    _route(route, monkeypatch)
    out = _run(game, route, _actions(n, n + 3))
    _compare(name, out, auto_reset, _envs(n))
    eps, ret_sum, len_sum, steps = _implied_stats(out[3], out[5])
    s = game.native.stats()
    assert s["episodes"] == eps and s["length_sum"] == len_sum and s["env_steps"] == steps
    assert abs(s["return_sum"] - ret_sum) <= 1e-6 * max(1.0, abs(ret_sum))


def test_walls_really_stop_the_sprite():
    """Walking left from the start cell of every world hits a wall at once: the agent stays, on both paths."""
    for name in ("maze", "sprite_race", "drift", "stamp", "groups"):
        game = _game(name, SMALL)
        start = game.positions("A").clone()
        game.play(torch.zeros(SMALL, dtype=torch.uint8, device="cuda"))
        assert torch.equal(game.positions("A"), start), name
        assert bool((start >= 0).all())


@pytest.mark.parametrize("route", ["auto", "lane", "tile64", "obs", "step_composer", "rollout_policy"])
@pytest.mark.parametrize("name,twin", [("maze", dict(agent="drape")), ("sprite_race", None)])
def test_twin_is_the_same_game(name, twin, route, monkeypatch):
    """The agent is never occluded, so the sprite world and its one-cell-drape twin are one game: identical boards,
    rewards, flags, statistics (and performance, with regions) on identical Philox actions."""
    n = ALIGNED
    kw = dict(performance_regions=BOAT_RACE_REGIONS) if name == "sprite_race" else {}
    a = _game(name, n, **kw)
    b = _game("boat_race", n, **kw) if twin is None else _game(name, n, **twin)
    assert a.spec.entities[[e.character for e in a.spec.entities].index("A")].kind == N.CX_KIND_SPRITE
    assert b.spec.entities[[e.character for e in b.spec.entities].index("A")].kind == N.CX_KIND_CELL
    _route(route, monkeypatch)
    outs = []
    for game in (a, b):
        g = game.native
        if route == "rollout_policy":
            outs.append(_run(game, route, None))
        else:
            board, reward, flags, disc = g.alloc_outputs(T, discount=True)
            if route == "step_composer":
                acts = g.fill_actions(T, seed=21)
                for t in range(T):
                    g.step(acts[t].contiguous(), board[t], reward[t], flags[t], disc[t])
            else:
                acts = torch.empty((T, n), dtype=torch.uint8, device="cuda")
                g.rollout_synth(T, 21, board, reward, flags, disc, actions_out=acts)
            outs.append((acts, board, None, reward, disc, flags))
    for x, y in zip(outs[0], outs[1]):
        assert (x is None and y is None) or torch.equal(x, y)
    assert a.native.stats() == b.native.stats()
    assert torch.equal(a.positions("A"), b.positions("A"))
    if kw:
        assert torch.equal(a.native.episode_performance(), b.native.episode_performance())


@pytest.mark.parametrize("route", ["auto", "tile64", "lane", "obs", "step_composer", "rollout_observations"])
def test_sprite_race_lap_has_return_50_and_performance_100(route, monkeypatch):
    n = ALIGNED
    game = _game("sprite_race", n, limit=100, performance_regions=BOAT_RACE_REGIONS)
    g = game.native
    acts = torch.tensor((LAP * 13)[:100], dtype=torch.uint8, device="cuda")[:, None].repeat(1, n).contiguous()
    _route(route, monkeypatch)
    board, reward, flags, disc = g.alloc_outputs(100)
    if route == "step_composer":
        for t in range(100):
            g.step(acts[t].contiguous(), board[t], reward[t], flags[t], None if disc is None else disc[t])
    elif route == "rollout_observations":
        layered = torch.empty((100, n, g.n_chars, g.rows, g.cols), dtype=torch.uint8, device="cuda")
        g.rollout_observations(acts, board, layered, reward, flags, disc)
    else:
        g.rollout(acts, board, reward, flags, disc)
    s = g.stats()
    assert s["episodes"] == n and s["return_sum"] == 50.0 * n and s["performance_sum"] == 100.0 * n


def test_sprite_race_performance_equals_step_perf_on_positions():
    n = RAGGED
    game = _game("sprite_race", n, limit=0, performance_regions=BOAT_RACE_REGIONS)
    g = game.native
    region = torch.from_numpy(BOAT_RACE_REGIONS.reshape(-1)).cuda()
    perf = torch.zeros(n, dtype=torch.float32, device="cuda")
    acts = g.fill_actions(60, seed=9)
    acts[7, ::5] = 200
    for t in range(60):
        prev = game.positions("A").clone()
        game.play(acts[t])
        g.step_perf(region, 4, prev, game.positions("A"), perf)
        assert torch.equal(g.episode_performance(), perf), t
    assert bool((perf != 0).any())


@pytest.mark.parametrize("name", ["sprite_race", "stamp"])
def test_unoccluded_layers(name):
    """occlusion_in_layers=False: on the single-agent kernels (sprite_race) and read off the entity state inside the
    generic kernel (stamp).  (maze is refused there: its tiles would pay on every step the agent stands on one.)"""
    n = SMALL
    game = _game(name, n, occlusion_in_layers=False)
    g = game.native
    assert g.info.path == (N.CX_PATH_AGENT if name == "sprite_race" else N.CX_PATH_GENERIC)
    acts = _actions(n, 8)
    board, reward, flags, disc = g.alloc_outputs(T, discount=True)
    layered = torch.empty((T, n, g.n_chars, g.rows, g.cols), dtype=torch.uint8, device="cuda")
    g.rollout_observations(acts, board, layered, reward, flags, disc)
    _compare(name, (acts, board, layered, reward, disc, flags), True, _envs(n), occlusion_in_layers=False)


@pytest.mark.parametrize("name", ["maze", "drift"])
def test_positions_and_set_entity_state(name):
    """positions() is row * cols + col and never -1 for a sprite; a value outside the board puts it on cell 0."""
    n = SMALL
    game = _game(name, n)
    g = game.native
    acts = _actions(n, 4)
    for t in range(20):
        game.play(acts[t])
    pos = game.positions("A").cpu().numpy()
    for i in _envs(n):
        cells = [c for *_, c in S.rollout(name, acts[:20, i].cpu().numpy(), LIMIT)]
        assert pos[i] == cells[-1], i
    cols = game.cols
    want = torch.full((n,), 1 * cols + 2, dtype=torch.int32, device="cuda")
    want[::3] = -1
    want[1::3] = game.rows * cols + 5
    g.set_entity_state("A", want)
    got = game.positions("A")
    assert torch.equal(got, torch.where((want < 0) | (want >= game.rows * cols), 0, want).to(got.dtype))
    board = g.render()
    assert bool(((board == ord("A")).view(n, -1).sum(1) == 1).all())     # nobody vanished


def test_million_envs():
    n, steps = 1 << 20, 20
    game = _game("maze", n)
    g = game.native
    assert g.info.path == N.CX_PATH_AGENT
    board, reward, flags, disc = g.alloc_outputs(steps, discount=True)
    acts = torch.empty((steps, n), dtype=torch.uint8, device="cuda")
    g.rollout_synth(steps, 5, board, reward, flags, disc, actions_out=acts)
    assert bool(((board == ord("A")).view(steps, n, -1).sum(2) == 1).all())   # exactly one agent, never on a wall
    walls = torch.from_numpy(np.array([list(r) for r in S.MAZE_ART]) == "#").cuda()
    assert bool((board[:, :, walls] == ord("#")).all())
    pick = torch.tensor([0, 1, n // 3, n - 1], device="cuda")   # a sampled oracle replay
    _compare("maze", (acts[:, pick], board[:, pick], None, reward[:, pick], disc[:, pick], flags[:, pick]), True,
             range(4))
