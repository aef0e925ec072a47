"""Games with key-locked doors (CX_KIND_DOOR) on the GPU, against the door oracle (tests/helpers/door_oracle.py, unpinned
by the reference) frame for frame: board, layers, reward, discount, flags and the items each env still holds, through
every route that runs pickup games; the doors each env shows after reset and render; statistics; a million envs."""
import numpy as np
import pytest
import torch

from campx_b200 import things
from campx_b200.ascii_art import Partial, ascii_art_to_game
from campx_b200.vector_env import VectorEnv
from examples.generality_worlds import Exit
from examples.worlds import DOORKEY_ART, Coin, Door, Walker, make_world
from tests.helpers import door_oracle as O
from tests.test_gpu_pickups import ROUTES

pytestmark = pytest.mark.gpu
T, LIMIT = 100, 40
DOOR_CELL, KEY_CELL = (2, 4), (3, 2)            # of DOORKEY_ART
NEXT_TO_DOOR = ['#########',                    # the key lies next to the door: taken, then passed on the next step
                '#A  #   #',
                '#  kD   #',
                '#   #  E#',
                '#########']
_GAMES = {}


def _game(n, auto_reset, two=False, art=None):
    key = (n, auto_reset, two, None if art is None else tuple(art))
    if key not in _GAMES:
        kw = dict(num_envs=n, max_episode_steps=LIMIT, auto_reset=auto_reset, track_returns=True)
        if art is None:
            g = make_world('doorkey2' if two else 'doorkey', **kw)
        else:
            g = ascii_art_to_game(art, ' ', drapes={'A': Partial(Walker, walls='#D'), 'D': Door, 'E': Partial(Exit, 10),
                                                    'k': Partial(Coin, value=0.0, pcontinue=None),
                                                    '#': things.FixedDrape},
                                  z_order='kDEA#', update_schedule='AEkD#', **kw)
        g.its_showtime()
        _GAMES[key] = g
    g = _GAMES[key]
    g.reset()
    return g


def _actions(n, seed, steps=T):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 5, size=(steps, n)).astype(np.uint8)
    a[rng.random((steps, n)) < 0.02] = 9          # now and then an action outside the set
    return torch.from_numpy(a).cuda()


def _run(g, route, acts):
    """-> (actions, board, layered or None, reward, discount, flags, items [T, n] or None) of T steps through `route`
    (the same routes as the pickup tests)"""
    nat, n, steps = g.native, g.num_envs, acts.shape[0]
    if route in ("rollout", "rollout_synth", "rollout_observations"):
        board, reward, flags, disc = nat.alloc_outputs(steps, discount=True)
        layered = None
        if route == "rollout":       # two launches
            cut = steps * 3 // 5
            for lo, hi in ((0, cut), (cut, steps)):
                nat.rollout(acts[lo:hi].contiguous(), board[lo:hi], reward[lo:hi], flags[lo:hi], disc[lo:hi])
        elif route == "rollout_synth":
            acts = torch.empty((steps, n), dtype=torch.uint8, device="cuda")
            nat.rollout_synth(steps, 77, board, reward, flags, disc, actions_out=acts)
        else:
            layered = torch.empty((steps, n, nat.n_chars, g.rows, g.cols), dtype=torch.uint8, device="cuda")
            nat.rollout_observations(acts, board, layered, reward, flags, disc)
        return acts, board, layered, reward, disc, flags, None
    boards, lays, rews, discs, flgs, items = [], [], [], [], [], []
    for t in range(steps):
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


def _envs(n, board, door=DOOR_CELL):
    """a few fixed envs, and the first two whose door opened during the run"""
    fixed = {0, 1, n // 2, n - 1} | ({31, 32, 63, 4096} if n > 64 else set(range(n)))
    opened = torch.nonzero((board[:, :, door[0], door[1]] != ord('D')).any(0)).view(-1)[:2].tolist()
    return sorted(i for i in fixed | set(opened) if i < n)


def _compare(out, auto_reset, two=False, envs=None, art=None):
    acts, board, layered, reward, disc, flags, items = (None if x is None else x.cpu().numpy() for x in out)
    for i in envs:
        for t, (b, lay, r, d, f, it) in enumerate(O.rollout(acts[:, i], two, LIMIT, auto_reset, art)):
            ctx = (i, t, int(acts[t, i]))
            assert np.array_equal(board[t, i], b), ctx
            if layered is not None:
                assert np.array_equal(layered[t, i], lay.astype(layered.dtype)), ctx
            assert float(reward[t, i]) == r and float(disc[t, i]) == d and int(flags[t, i]) == f, ctx
            if items is not None:
                assert int(items[t, i]) & ((1 << 64) - 1) == it, ctx


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("n", [1, 5, 64, 272, 4099])
@pytest.mark.parametrize("route", ROUTES)
def test_matches_the_oracle(route, n, auto_reset):
    g = _game(n, auto_reset)
    out = _run(g, route, _actions(n, n))
    envs = _envs(n, out[1])
    if n >= 64:          # random walks open the door somewhere ...
        assert any((out[1][:, i, DOOR_CELL[0], DOOR_CELL[1]] != ord('D')).any() for i in envs)
    if n >= 272:         # ... and some reach the exit
        assert bool(((out[5] & O.CX_FLAG_TERMINATED) != 0).any())
    _compare(out, auto_reset, envs=envs)


@pytest.mark.parametrize("route", ["step", "rollout", "rollout_observations", "play"])
def test_two_keys_two_doors(route):
    n = 4099
    g = _game(n, True, two=True)
    out = _run(g, route, _actions(n, 3))
    board = out[1]
    both = (board[:, :, 2, 4] != ord('D')) & (board[:, :, 2, 8] != ord('d'))
    assert bool(both.any())                        # some env opened both doors
    envs = sorted(set(_envs(n, board)) | set(torch.nonzero(both.any(0)).view(-1)[:2].tolist()))
    _compare(out, True, two=True, envs=envs)


def _scripted(g, route, script):
    acts = torch.tensor(script, dtype=torch.uint8, device="cuda")[:, None].repeat(1, g.num_envs).contiguous()
    return _run(g, route, acts)


@pytest.mark.parametrize("route", [r for r in ROUTES if r != "rollout_synth"])
def test_scripted_episode(route):
    """Into the closed door (blocked), take the key (the door opens in that frame), through the door, to the exit; the
    auto reset closes the door again.  Then: the key next to the door, taken, and the door passed on the next step."""
    down, right, left, up, stay = 3, 1, 0, 2, 4
    script = [down, right, right, right, down, left, left, up, right, right, right, right, right, down, right, stay]
    g = _game(32, True)
    out = _scripted(g, route, script)
    _compare(out, True, envs=[0, 31])
    board, reward, flags = out[1].cpu().numpy()[:, 0], out[3].cpu().numpy()[:, 0], out[5].cpu().numpy()[:, 0]
    dr, dc = DOOR_CELL
    assert chr(board[3, 2, 3]) == 'A' and chr(board[3, dr, dc]) == 'D'           # blocked by the closed door
    assert chr(board[4, dr, dc]) == 'D' and chr(board[5, dr, dc]) == ' '         # the key taken at step 5: open
    assert chr(board[5, KEY_CELL[0], KEY_CELL[1]]) == 'A'
    assert chr(board[10, dr, dc]) == 'A'                                         # through the door
    assert reward[14] == 10 and flags[14] & O.CX_FLAG_TERMINATED                 # the exit
    assert chr(board[15, dr, dc]) == 'D' and chr(board[15, KEY_CELL[0], KEY_CELL[1]]) == 'k'   # reset: closed again

    g = _game(32, True, art=NEXT_TO_DOOR)
    out = _scripted(g, route, [down, right, right, right, right])
    _compare(out, True, envs=[0, 31], art=NEXT_TO_DOOR)
    board = out[1].cpu().numpy()[:, 0]
    assert chr(board[2, 2, 3]) == 'A' and chr(board[2, dr, dc]) == ' '          # key taken: open in the same frame
    assert chr(board[3, dr, dc]) == 'A'                                          # ... and passed on the next step


def test_reset_render_and_door_state():
    n = 4099
    g = _game(n, False)
    _run(g, "rollout", _actions(n, 7))
    nat = g.native
    before = nat.pickups()
    doors = nat.doors()
    assert doors.shape == (n, 1) and doors.any() and not doors.all()
    assert torch.equal(doors[:, 0], g.door_open('D')) and torch.equal(doors[:, 0], before == 0)
    board = torch.empty((n, g.rows, g.cols), dtype=torch.uint8, device="cuda")
    for dtype in (torch.uint8, torch.float32):
        layered = torch.empty((n, nat.n_chars, g.rows, g.cols), dtype=dtype, device="cuda")
        nat.render_observations(board, layered)
        shut = board[:, DOOR_CELL[0], DOOR_CELL[1]] == ord('D')
        assert torch.equal(shut, ~g.door_open('D'))
        assert torch.equal(layered, nat.layers_from_board(board).to(dtype))
    assert torch.equal(nat.render(), board)
    mask = (torch.arange(n, device="cuda") % 3 == 0).to(torch.uint8)
    nat.reset(mask)
    after = nat.doors()[:, 0]
    assert not after[mask.bool()].any() and torch.equal(after[~mask.bool()], doors[~mask.bool(), 0])
    nat.render_observations(board, layered)
    assert torch.equal(board[:, DOOR_CELL[0], DOOR_CELL[1]] == ord('D'), ~after)
    nat.reset()
    assert not nat.doors().any() and bool((nat.render()[:, DOOR_CELL[0], DOOR_CELL[1]] == ord('D')).all())
    with pytest.raises(ValueError):
        g.door_open('k')
    with pytest.raises(ValueError):
        nat.entity_state('D')


def test_stats_equal_the_reward_and_flag_streams():
    n = 4099
    g = _game(n, True)
    acts, board, layered, reward, disc, flags, _ = _run(g, "rollout", _actions(n, 11))
    r, f = reward.cpu().numpy().astype(np.float64), flags.cpu().numpy()
    eps = ret_sum = len_sum = 0.0
    ret, steps = np.zeros(n), np.zeros(n)
    for t in range(T):
        counts = (f[t] & (O.CX_FLAG_BAD_ACTION | O.CX_FLAG_ALREADY_OVER)) == 0
        ret += np.where(counts, np.float32(r[t]), 0)
        steps += counts
        done = counts & ((f[t] & (O.CX_FLAG_TERMINATED | O.CX_FLAG_TRUNCATED)) != 0)
        eps += done.sum()
        ret_sum += ret[done].sum()
        len_sum += steps[done].sum()
        ret[done], steps[done] = 0, 0
    s = g.episode_stats()
    assert s["episodes"] == eps and s["length_sum"] == len_sum and s["env_steps"] == n * T
    assert abs(s["return_sum"] - ret_sum) < 1e-6 * max(1.0, ret_sum)
    assert (f & O.CX_FLAG_TERMINATED).any()


def test_million_envs():
    n, steps = 1 << 20, 20
    g = _game(n, True)
    nat = g.native
    board, reward, flags, disc = nat.alloc_outputs(steps, discount=True)
    acts = torch.empty((steps, n), dtype=torch.uint8, device="cuda")
    nat.rollout_synth(steps, 5, board, reward, flags, disc, actions_out=acts)
    # every frame shows the door closed exactly while the key lies on the board (the agent only stands on a taken key)
    shut = board[:, :, DOOR_CELL[0], DOOR_CELL[1]] == ord('D')
    assert torch.equal(shut, board[:, :, KEY_CELL[0], KEY_CELL[1]] == ord('k'))
    assert bool((~shut).any())
    opened = torch.nonzero((~shut).any(0)).view(-1)
    pick = torch.cat([torch.tensor([0, 1, n // 3, n - 1], device="cuda"), opened[:2], opened[-2:]])
    sub = (acts[:, pick], board[:, pick], None, reward[:, pick], disc[:, pick], flags[:, pick], None)
    _compare(sub, True, envs=range(len(pick)))


def test_vector_env_board_policy_and_what_is_refused():
    env = VectorEnv(make_world('doorkey', num_envs=64, max_episode_steps=LIMIT))
    first = env.reset()
    assert (first[:, DOOR_CELL[0], DOOR_CELL[1]] == ord('D')).all()
    for a in (3, 1, 1, 1):                              # down, then right into the closed door
        obs, reward, terminated, truncated, info = env.step(torch.full((64,), a, dtype=torch.uint8, device="cuda"))
    assert (obs[:, 2, 3] == ord('A')).all() and not terminated.any()
    g = _game(256, True)
    nat = g.native
    board = _run(g, "rollout", _actions(256, 2, steps=12))[1][-1].contiguous()
    feat = nat.n_chars * nat.cells
    torch.manual_seed(1)
    w1t, b1 = torch.randn((feat, 32), device="cuda"), torch.randn(32, device="cuda")
    w2, b2 = torch.randn((5, 32), device="cuda"), torch.randn(5, device="cuda")
    outs = [(torch.empty(256, dtype=torch.uint8, device="cuda"), torch.empty(256, device="cuda"),
             torch.empty((256, 5), device="cuda")) for _ in range(2)]
    step = torch.full((1,), 7, dtype=torch.int64, device="cuda")
    nat.policy_sample_board(board, w1t, b1, w2, b2, 11, step=step, step_offset=3, out=outs[0][0], logp=outs[0][1],
                            logits_out=outs[0][2])
    planes = nat.layers_from_board(board, dtype=torch.float32).view(256, -1)
    nat.policy_sample(planes, w1t, b1, w2, b2, 11, step=step, step_offset=3, out=outs[1][0], logp=outs[1][1],
                      logits_out=outs[1][2])
    assert all(torch.equal(x, y) for x, y in zip(*outs))
    states = torch.empty((3, 256, feat), device="cuda")
    a, r, f = (torch.empty((2, 256), dtype=dt, device="cuda") for dt in (torch.uint8, torch.float32, torch.uint8))
    with pytest.raises(NotImplementedError):
        nat.rollout_policy(2, w1t, b1, w2, b2, 0, states, a, r, f)
    assert nat.info.n_pickups == 1
