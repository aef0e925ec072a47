"""Games with collectible items (CX_KIND_PICKUP) on the GPU, against the pickup oracle (tests/helpers/pickup_oracle.py,
unpinned by the reference) frame for frame: board, layers, reward, discount, flags and the items each env still holds,
through every route that runs them."""
import numpy as np
import pytest
import torch

from campx_b200 import _native as N
from campx_b200 import things
from campx_b200.ascii_art import Partial, ascii_art_to_game
from campx_b200.vector_env import VectorEnv
from examples.worlds import COINS_ART, Coin, Walker, make_world
from tests.helpers import pickup_oracle as P

pytestmark = pytest.mark.gpu
T, LIMIT = 100, 30
ALL = (1 << 10) - 1
ROUTES = ["step", "rollout", "rollout_synth", "rollout_observations", "step_observations_f32", "play"]
SMALL_ART = ['#####', '#A$$#', '#$  #', '#####']   # three coins: random walks take them all within T steps
_GAMES = {}


def _game(n, auto_reset, schedule='A$#', pcontinue=0.0, art=COINS_ART):
    key = (n, auto_reset, schedule, pcontinue, tuple(art))
    if key not in _GAMES:
        g = ascii_art_to_game(art, ' ', drapes={'A': Partial(Walker, walls='#'), '$': Partial(Coin, pcontinue=pcontinue),
                                                '#': things.FixedDrape},
                              z_order='$A#', update_schedule=schedule, num_envs=n, max_episode_steps=LIMIT,
                              auto_reset=auto_reset, track_returns=True)
        g.its_showtime()
        _GAMES[key] = g
    g = _GAMES[key]
    g.reset()
    return g


def _actions(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 5, size=(T, n)).astype(np.uint8)
    a[rng.random((T, n)) < 0.02] = 9          # now and then an action outside the set
    return torch.from_numpy(a).cuda()


def _run(g, route, acts):
    """-> (actions, board, layered or None, reward, discount, flags, items [T, n]) of T steps through `route`"""
    nat, n = g.native, g.num_envs
    items = []
    if route in ("rollout", "rollout_synth", "rollout_observations"):
        board, reward, flags, disc = nat.alloc_outputs(T, discount=True)
        layered = None
        if route == "rollout":       # two launches, 60 + 40 steps
            for lo, hi in ((0, 60), (60, T)):
                nat.rollout(acts[lo:hi].contiguous(), board[lo:hi], reward[lo:hi], flags[lo:hi], disc[lo:hi])
        elif route == "rollout_synth":
            acts = torch.empty((T, n), dtype=torch.uint8, device="cuda")
            nat.rollout_synth(T, 77, board, reward, flags, disc, actions_out=acts)
        else:
            layered = torch.empty((T, n, nat.n_chars, g.rows, g.cols), dtype=torch.uint8, device="cuda")
            nat.rollout_observations(acts, board, layered, reward, flags, disc)
        return acts, board, layered, reward, disc, flags, None
    boards, lays, rews, discs, flgs = [], [], [], [], []
    for t in range(T):
        if route == "play":
            obs, reward, discount = g.play(acts[t])
            boards.append(obs.board.clone())
            lays.append(obs.layered_board.clone())
            rews.append(reward.clone())
            discs.append(discount.clone())
            flgs.append(g.flags.clone())
        else:
            board, reward, flags, disc = nat.alloc_outputs(None, discount=True)
            lay = None
            if route == "step":
                nat.step(acts[t].contiguous(), board, reward, flags, disc)
            else:
                lay = torch.empty((n, nat.n_chars, g.rows, g.cols), dtype=torch.float32, device="cuda")
                nat.step_observations(acts[t].contiguous(), board, lay, reward, flags, disc)
            boards.append(board)
            lays.append(lay)
            rews.append(reward)
            discs.append(disc)
            flgs.append(flags)
        items.append(nat.pickups())
    layered = None if lays[0] is None else torch.stack(lays)
    return (acts, torch.stack(boards), layered, torch.stack(rews), torch.stack(discs), torch.stack(flgs),
            torch.stack(items))


def _envs(n):
    return sorted(i for i in {0, 1, n // 2, n - 1} | ({31, 32, 63, 4096} if n > 64 else set(range(n))) if i < n)


def _compare(out, n, auto_reset, schedule='A$#', envs=None, pcontinue=0.0, art=COINS_ART):
    acts, board, layered, reward, disc, flags, items = (None if x is None else x.cpu().numpy() for x in out)
    for i in (envs if envs is not None else _envs(n)):
        for t, (b, lay, r, d, f, it) in enumerate(P.rollout(acts[:, i], schedule, LIMIT, auto_reset, pcontinue, art)):
            ctx = (i, t, int(acts[t, i]))
            assert np.array_equal(board[t, i], b), ctx
            if layered is not None:
                assert np.array_equal(layered[t, i], lay.astype(layered.dtype)), ctx
            assert float(reward[t, i]) == r and float(disc[t, i]) == d and int(flags[t, i]) == f, ctx
            if items is not None:
                assert int(items[t, i]) & ((1 << 64) - 1) == it, ctx
    return acts, reward, flags


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("n", [1, 5, 64, 272, 4099])
@pytest.mark.parametrize("route", ROUTES)
def test_matches_the_oracle(route, n, auto_reset):
    g = _game(n, auto_reset)
    _compare(_run(g, route, _actions(n, n)), n, auto_reset)


@pytest.mark.parametrize("route", ["step", "rollout", "rollout_observations"])
def test_pickups_updating_before_the_agent(route):
    g = _game(272, True, schedule='$A#')
    _compare(_run(g, route, _actions(272, 5)), 272, True, schedule='$A#')


def test_stats_equal_the_reward_and_flag_streams():
    n = 4099
    g = _game(n, True, art=SMALL_ART)
    acts, board, layered, reward, disc, flags, _ = _run(g, "rollout", _actions(n, 11))
    r, f = reward.cpu().numpy().astype(np.float64), flags.cpu().numpy()
    eps = ret_sum = len_sum = 0.0
    ret, steps = np.zeros(n), np.zeros(n)
    for t in range(T):
        counts = (f[t] & (P.CX_FLAG_BAD_ACTION | P.CX_FLAG_ALREADY_OVER)) == 0
        ret += np.where(counts, np.float32(r[t]), 0)
        steps += counts
        done = counts & ((f[t] & (P.CX_FLAG_TERMINATED | P.CX_FLAG_TRUNCATED)) != 0)
        eps += done.sum()
        ret_sum += ret[done].sum()
        len_sum += steps[done].sum()
        ret[done], steps[done] = 0, 0
    s = g.episode_stats()
    assert s["episodes"] == eps and s["length_sum"] == len_sum and s["env_steps"] == n * T
    assert abs(s["return_sum"] - ret_sum) < 1e-6 * max(1.0, ret_sum)
    assert eps > 0 and (f & P.CX_FLAG_TERMINATED).any()


def test_all_collected_carries_the_discount():
    n = 4099
    g = _game(n, True, pcontinue=0.25, art=SMALL_ART)
    out = _run(g, "rollout", _actions(n, 3))
    flags, disc = out[5].cpu().numpy(), out[4].cpu().numpy()
    term = (flags & P.CX_FLAG_TERMINATED) != 0
    assert term.any() and (disc[term] == np.float32(0.25)).all()
    _compare(out, n, True, envs=[int(np.argwhere(term)[0][1]), 0], pcontinue=0.25, art=SMALL_ART)


def test_reset_and_render_show_the_right_items():
    n = 4099
    g = _game(n, False)
    _run(g, "rollout", _actions(n, 7))
    nat = g.native
    before = nat.pickups()
    assert (before != ALL).any()
    board = torch.empty((n, g.rows, g.cols), dtype=torch.uint8, device="cuda")
    for dtype in (torch.uint8, torch.float32):
        layered = torch.empty((n, nat.n_chars, g.rows, g.cols), dtype=dtype, device="cuda")
        nat.render_observations(board, layered)
        assert torch.equal(board == ord('$'), g.pickup_curtain('$'))    # the agent never stands on a coin
        assert torch.equal(layered, nat.layers_from_board(board).to(dtype))
    assert torch.equal(nat.render(), board)
    mask = (torch.arange(n, device="cuda") % 3 == 0).to(torch.uint8)
    nat.reset(mask)
    after = nat.pickups()
    assert (after[mask.bool()] == ALL).all() and torch.equal(after[~mask.bool()], before[~mask.bool()])
    nat.reset()
    assert (nat.pickups() == ALL).all()
    nat.render_observations(board, layered)
    assert ((board == ord('$')).view(n, -1).sum(1) == 10).all()


def test_million_envs():
    n, steps = 1 << 20, 20
    g = _game(n, True)
    nat = g.native
    board, reward, flags, disc = nat.alloc_outputs(steps, discount=True)
    acts = torch.empty((steps, n), dtype=torch.uint8, device="cuda")
    nat.rollout_synth(steps, 5, board, reward, flags, disc, actions_out=acts)
    coins = (board == ord('$')).view(steps, n, -1).sum(2)
    left = torch.full((n,), 10, device="cuda")
    for t in range(steps):   # every paid step takes one coin from the board; an episode ends with none or at the limit
        assert ((reward[t] == 0) | (reward[t] == 1)).all()
        left = left - reward[t].long()
        assert torch.equal(coins[t], left)
        assert torch.equal((flags[t] & P.CX_FLAG_TERMINATED) != 0, left == 0)
        left = torch.where((flags[t] & (P.CX_FLAG_TERMINATED | P.CX_FLAG_TRUNCATED)) != 0, 10, left)
    bits = nat.pickups()
    pop = sum(((bits >> k) & 1) for k in range(10))
    assert torch.equal(pop, left)
    pick = torch.tensor([0, 1, n // 3, n - 1], device="cuda")   # a sampled oracle replay
    _compare((acts[:, pick], board[:, pick], None, reward[:, pick], disc[:, pick], flags[:, pick], None), 4, True,
             envs=range(4))


def test_vector_env_and_what_is_refused():
    env = VectorEnv(make_world('coins', num_envs=64, max_episode_steps=LIMIT))
    first = env.reset()
    assert ((first == ord('$')).view(64, -1).sum(1) == 10).all()
    right = torch.ones(64, dtype=torch.uint8, device="cuda")
    env.step(right)
    obs, reward, terminated, truncated, info = env.step(right)   # '#A $': two steps right take the first coin
    assert obs.shape == first.shape and (reward == 1).all() and not terminated.any()
    assert ((obs == ord('$')).view(64, -1).sum(1) == 9).all()
    g = _game(64, True)
    nat = g.native
    feat = nat.n_chars * nat.cells
    w1t, b1 = torch.zeros((feat, 8), device="cuda"), torch.zeros(8, device="cuda")
    w2, b2 = torch.zeros((5, 8), device="cuda"), torch.zeros(5, device="cuda")
    states = torch.empty((3, 64, feat), device="cuda")
    a, r, f = (torch.empty((2, 64), dtype=dt, device="cuda") for dt in (torch.uint8, torch.float32, torch.uint8))
    with pytest.raises(NotImplementedError):
        nat.rollout_policy(2, w1t, b1, w2, b2, 0, states, a, r, f)
    acts = nat.policy_sample_board(nat.render(), w1t, b1, w2, b2, 0)   # reads boards: works unchanged
    assert acts.shape == (64,)
    board = torch.empty((64, g.rows, g.cols), dtype=torch.uint8, device="cuda")
    with pytest.raises(NotImplementedError):
        nat.render_observations(board, torch.empty((64, nat.n_chars, g.rows, g.cols), dtype=torch.bfloat16,
                                                   device="cuda"))
    with pytest.raises(ValueError):
        nat.entity_state('$')
    assert nat.info.n_pickups == 10 and nat.info.path == N.CX_PATH_AGENT
