"""GPU parity through the public API (ascii_art_to_game -> Engine.its_showtime/play/rollout): the user-level
worlds of examples/worlds.py are compiled by the front end, run by the CUDA kernels through the C ABI
and compared with the golden fixtures (recorded from the reference) and the numpy oracle."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import campx_oracle as O
from examples.worlds import make_world as _make_reference_world, BOAT_RACE_REGIONS
from examples.generality_worlds import make_generality_world
from tests.helpers.policy_reference import philox4

pytestmark = pytest.mark.gpu

# the six reference worlds + the engine-generality worlds (z-order directives, sprite visibility, scrolling
# backdrop: SURVEY 8(f) row 3), whose fixtures were also recorded from the reference (oracle/gen_golden.py)
# and the "reach the goal" worlds (terminate_episode depends on the cell the agent reached)
WORLDS = ["boat_race", "demo1", "demo2", "demo3", "demo4", "hello", "zswap", "ghost", "scroll", "goal", "goal2"]


def make_world(name, **kw):
    if name in O.GENERALITY_WORLDS + O.GOAL_WORLDS:
        return make_generality_world(name, **kw)
    return _make_reference_world(name, **kw)


def golden_path(golden_dir, world):
    extra = world in O.GENERALITY_WORLDS + O.GOAL_WORLDS
    return os.path.join(golden_dir, ("generality_" if extra else "") + world + ".json")


def board_str(b):
    return "".join(chr(int(v)) for v in b.reshape(-1).tolist())


def ref_action(world, a):
    """The action object a reference user passes for index a (boat_race.py:26; notebooks)."""
    if world in ("hello", "zswap", "ghost"):
        return int(a)
    onehot = [0] * 5
    onehot[a] = 1
    return torch.FloatTensor(onehot) if world in ("boat_race", "demo4", "scroll", "goal", "goal2") else onehot


@pytest.mark.parametrize("world", WORLDS)
def test_single_env_drop_in_matches_golden(golden_dir, world):
    """num_envs=None: reference shapes, reference action objects, reference error behaviour."""
    with open(golden_path(golden_dir, world)) as f:
        fx = json.load(f)
    for ep in fx["episodes"][:3]:
        game = make_world(world)
        obs, reward, discount = game.its_showtime()
        f0 = ep["frames"][0]
        assert obs.board.shape == (game.rows, game.cols)
        assert board_str(obs.board.cpu()) == f0["board"] and reward is None and discount == 1.0
        for t, a in enumerate(ep["actions"]):
            obs, reward, discount = game.play(ref_action(world, a))
            want = ep["frames"][t + 1]
            assert board_str(obs.board.cpu()) == want["board"]
            assert reward == want["reward"] and discount == want["discount"]
            for ch in want["layers"]:
                got = "".join(str(int(v)) for v in obs.layers[ch].cpu().reshape(-1).tolist())
                assert got == want["layers"][ch]
            assert obs.layered_board.shape == (len(want["layers"]), game.rows, game.cols)
            board2, layers2, layered2 = obs                    # unpacks like the reference's namedtuple
            assert board2 is obs.board and layered2 is obs.layered_board
        if ep["error_after"]:
            with pytest.raises(RuntimeError) as ei:
                game.play(ref_action(world, 0))
            assert str(ei.value) == ep["error_after"]          # engine.py:149-151


def test_play_before_showtime_and_bad_actions():
    game = make_world("boat_race")
    with pytest.raises(RuntimeError):
        game.play(torch.FloatTensor([0, 1, 0, 0, 0]))
    game.its_showtime()
    with pytest.raises(RuntimeError):
        game.its_showtime()                                    # engine.py:513
    with pytest.raises(ValueError):
        game.play(torch.FloatTensor([0, 1, 1, 0, 0]))          # boat_race.py:48: exactly one action
    with pytest.raises(ValueError):
        game.play(7)


def test_batched_actions_that_are_not_actions_are_flagged_not_guessed():
    """ADVICE r1: a batched one-hot row with no 1, several 1s or fractional entries used to be argmax-ed silently, and
    int64 indices >= 256 wrapped into the action set.  Both now leave the env untouched and raise CX_FLAG_BAD_ACTION
    (the single-env mode, like the reference's `assert sum(act) == 1`, raises)."""
    from campx_b200 import _native as N
    n = 64
    game = make_world("boat_race", num_envs=n)
    obs, _, _ = game.its_showtime()
    first = obs.board.clone()
    onehot = torch.zeros((n, 5), device="cuda")
    onehot[:, 1] = 1                                           # everybody: right
    onehot[3] = 0                                              # no action at all
    onehot[5, 3] = 1                                           # two actions
    onehot[7] = torch.tensor([0, 0.5, 0.5, 0, 0])              # fractional
    obs, reward, _ = game.play(onehot)
    bad = (game.flags & N.CX_FLAG_BAD_ACTION) != 0
    assert bad.nonzero().flatten().tolist() == [3, 5, 7] and game.bad_action_count() == 3
    assert torch.equal(obs.board[bad], first[bad]) and bool((reward[bad] == 0).all())
    assert bool((obs.board[~bad] != first[~bad]).flatten(1).any(dim=1).all())       # the others moved
    idx = torch.full((n,), 1, dtype=torch.int64, device="cuda")
    idx[2], idx[4] = 257, -1                                   # 257 must not wrap to action 1, -1 not to 255 & co
    before = obs.board.clone()
    obs, reward, _ = game.play(idx)
    bad = (game.flags & N.CX_FLAG_BAD_ACTION) != 0
    assert bad.nonzero().flatten().tolist() == [2, 4] and torch.equal(obs.board[bad], before[bad])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_games_on_a_second_device():
    """ADVICE r1: the dynamic-shared-memory cap is a per-DEVICE function attribute; a process that had configured it on
    cuda:0 used to launch unconfigured on cuda:1."""
    a = make_world("boat_race", num_envs=1 << 16, device="cuda:0")
    a.its_showtime()
    acts = a.native.fill_actions(8, seed=1)
    ref = a.rollout(acts)
    b = make_world("boat_race", num_envs=1 << 16, device="cuda:1")
    b.its_showtime()
    with torch.cuda.device(1):
        got = b.rollout(acts.to("cuda:1"))
        lay = b.rollout_observations(acts.to("cuda:1"))[1]
    assert torch.equal(ref[0], got[0].to("cuda:0")) and torch.equal(ref[1], got[1].to("cuda:0"))
    assert lay.device.index == 1
    h = make_world("hello", num_envs=4096, device="cuda:1")
    h.its_showtime()
    with torch.cuda.device(1):
        hb = h.rollout(h.native.fill_actions(4, seed=2))[0]
    assert hb.device.index == 1 and int((hb == ord("@")).sum()) > 0


@pytest.mark.parametrize("world", WORLDS)
def test_batched_play_matches_oracle(world):
    n, T, limit = 48, 40, 15
    game = make_world(world, num_envs=n, max_episode_steps=limit)
    obs, reward, discount = game.its_showtime()
    assert obs.board.shape == (n, game.rows, game.cols) and reward is None
    assert torch.equal(discount, torch.ones(n, device=discount.device))
    rng = np.random.Generator(np.random.PCG64(99))
    acts = rng.integers(0, 5, size=(T, n)).astype(np.uint8)
    if world == "hello":
        acts[(acts == 4) & (rng.random((T, n)) < 0.7)] = 1
    oracles = [O.rollout(world, acts[:, i], rebuild_on_done=True, max_episode_steps=limit) for i in range(n)]
    for t in range(T):
        if world in ("boat_race", "demo4", "scroll") and t % 2:   # one-hot float batch, as the reference's worlds take
            a = torch.nn.functional.one_hot(torch.from_numpy(acts[t]).long(), 5).float().cuda()
        else:
            a = torch.from_numpy(acts[t]).cuda()
        obs, reward, discount = game.play(a)
        b, r, d = obs.board.cpu().numpy(), reward.cpu().numpy(), discount.cpu().numpy()
        none = game.reward_is_none.cpu().numpy()
        lay = obs.layered_board.cpu().numpy()
        for i in range(n):
            o, rew, dsc, term, trunc, eng = next(oracles[i])
            assert np.array_equal(b[i], np.asarray(o.board).astype(np.uint8)), (world, i, t)
            assert (rew is None) == bool(none[i])
            if rew is not None:
                assert float(rew) == float(r[i])
            assert float(dsc) == float(d[i])
            assert np.array_equal(lay[i], np.asarray(o.layered_board).astype(np.uint8))
            for ch in game.characters:
                assert np.array_equal(obs.layers[ch][i].cpu().numpy(), o.layers[ch])


def test_positions_and_step_perf_boat_race():
    """Agent cells (positions) and the hidden safety performance (boat_race.py:117-151)."""
    n, T = 64, 30
    game = make_world("boat_race", num_envs=n)
    game.its_showtime()
    rng = np.random.Generator(np.random.PCG64(5))
    acts = rng.integers(0, 5, size=(T, n)).astype(np.uint8)
    region = torch.from_numpy(BOAT_RACE_REGIONS.reshape(-1).copy()).cuda()
    perf = torch.zeros(n, dtype=torch.float32, device="cuda")
    worlds = [O.World("boat_race") for _ in range(n)]
    want_perf = np.zeros(n)
    ring = [(1, 1), (1, 2), (1, 3), (2, 3), (3, 3), (3, 2), (3, 1), (2, 1)]     # clockwise
    prev = game.positions("A")
    for t in range(T):
        game.play(torch.from_numpy(acts[t]).cuda())
        nxt = game.positions("A")
        game.native.step_perf(region, 4, prev, nxt, perf)
        p, q = prev.cpu().numpy(), nxt.cpu().numpy()
        for i in range(n):
            worlds[i].step(int(acts[t, i]))
            mask = worlds[i].engine.things["A"].curtain
            assert int(np.flatnonzero(mask.reshape(-1))[0]) == q[i]
            ip, iq = ring.index((p[i] // 5, p[i] % 5)), ring.index((q[i] // 5, q[i] % 5))
            want_perf[i] += {1: 1, 7: -1}.get((iq - ip) % 8, 0)
        prev = nxt
    assert np.array_equal(perf.cpu().numpy(), want_perf)


def test_preset_lap_return_and_performance():
    """examples/README.md:31-33: a clockwise lap pays 2,-1,... ; select_action_preset (boat_race.py:154-184)."""
    preset = [1, 1, 3, 3, 0, 0, 2, 2, 3, 3, 1, 1, 2, 2, 0, 0, 0, 4, 4, 4]
    n = 32
    game = make_world("boat_race", num_envs=n, track_returns=True)
    game.its_showtime()
    acts = torch.tensor(preset, dtype=torch.uint8).repeat(n, 1).t().contiguous().cuda()
    boards, rewards, discounts, flags = game.rollout(acts)
    want = [2, -1, 2, -1, 2, -1, 2, -1, 0, -1, 0, -1, 0, -1, 0, -1, -1, -1, -1, -1]
    assert rewards.cpu().t().tolist() == [want] * n
    assert discounts is None and int(flags.max()) == 0
    steps, returns = game.native.episode_state()
    assert steps.tolist() == [20] * n and returns.tolist() == [float(sum(want))] * n


def test_rollout_equals_play_and_sharding_is_deterministic():
    """N-GPU run == concatenation of single-GPU runs on the same per-env action streams: with envs
    independent and Philox actions keyed by global env id, two half-batches reproduce one full batch."""
    n, T = 512, 50
    full = make_world("boat_race", num_envs=n, max_episode_steps=20, track_returns=True)
    full.its_showtime()
    a_full = full.native.fill_actions(T, seed=543, env_offset=0)
    out_full = full.rollout(a_full)
    halves = []
    for r in range(2):
        g = make_world("boat_race", num_envs=n // 2, max_episode_steps=20, track_returns=True)
        g.its_showtime()
        a = g.native.fill_actions(T, seed=543, env_offset=r * (n // 2))
        assert torch.equal(a, a_full[:, r * (n // 2):(r + 1) * (n // 2)])
        halves.append((g, g.rollout(a)))
    for k in (0, 1, 3):
        cat = torch.cat([h[1][k] for h in halves], dim=1)
        assert torch.equal(cat, out_full[k])
    s = full.episode_stats()
    hs = [h[0].episode_stats() for h in halves]
    for key in ("episodes", "return_sum", "return_sumsq", "length_sum", "env_steps"):
        assert s[key] == hs[0][key] + hs[1][key]
    assert s["return_max"] == max(h["return_max"] for h in hs)
    # play() step by step == fused rollout
    step = make_world("boat_race", num_envs=n, max_episode_steps=20, track_returns=True)
    step.its_showtime()
    for t in range(T):
        obs, reward, _ = step.play(a_full[t])
        assert torch.equal(obs.board, out_full[0][t]) and torch.equal(reward, out_full[1][t])
        assert torch.equal(step.flags, out_full[3][t])


def test_philox_actions_match_host_reference():
    """cx_fill_actions is counter-based: any (env, t) is regenerable on the host."""
    game = make_world("boat_race", num_envs=64)
    game.its_showtime()
    a = game.native.fill_actions(7, seed=543, env_offset=1000, t0=3).cpu().numpy()
    for t in range(7):
        for i in (0, 1, 2, 3, 17, 63):
            g = 1000 + i
            assert a[t, i] == (philox4(543, g >> 2, 3 + t)[g & 3] * 5) >> 32
    hist = np.bincount(game.native.fill_actions(200, seed=1).cpu().numpy().reshape(-1), minlength=5) / (200 * 64)
    assert np.all(np.abs(hist - 0.2) < 0.02)


@pytest.mark.parametrize("world,n", [("boat_race", 1024), ("boat_race", 100), ("demo3", 512), ("hello", 96)])
def test_in_kernel_random_rollout_equals_fill_actions_plus_rollout(world, n):
    """cx_rollout_synth draws the actions inside the kernel from the same Philox stream."""
    T, seed, off, t0 = 37, 543, 4096, 11
    a = make_world(world, num_envs=n, max_episode_steps=20, track_returns=True)
    b = make_world(world, num_envs=n, max_episode_steps=20, track_returns=True)
    a.its_showtime()
    b.its_showtime()
    acts = a.native.fill_actions(T, seed=seed, env_offset=off, t0=t0)
    ra = a.rollout(acts)
    played = torch.empty_like(acts)
    rb = b.rollout_random(T, seed, env_offset=off, t0=t0, actions_out=played)
    assert torch.equal(played, acts)
    for x, y in zip(ra, rb):
        assert (x is None and y is None) or torch.equal(x, y)
    a.native.fold_stats(), b.native.fold_stats()
    assert torch.equal(a.native.state, b.native.state)
    rc = b.rollout_random(3, seed, env_offset=off, t0=t0 + T)           # without writing the actions out
    rd = a.rollout(a.native.fill_actions(3, seed=seed, env_offset=off, t0=t0 + T))
    assert torch.equal(rc[0], rd[0]) and torch.equal(rc[1], rd[1])
    with pytest.raises(ValueError):
        b.rollout_random(2, seed, env_offset=3)


def test_full_size_properties_boat_race():
    """2^20 envs x 64 steps: size-independent properties + a sampled oracle replay."""
    n, T = 1 << 20, 64
    game = make_world("boat_race", num_envs=n, max_episode_steps=100, track_returns=True)
    game.its_showtime()
    acts = game.native.fill_actions(T, seed=543)
    boards, rewards, discounts, flags = game.rollout(acts)
    flat = boards.view(T, n, 25)
    assert int((flat == ord("A")).sum(dim=2).min()) == 1 and int((flat == ord("A")).sum(dim=2).max()) == 1
    walls = torch.tensor([c == "#" for c in "".join(O.BOAT_RACE_ART)], device=flat.device)
    assert bool((flat[:, :, walls] == ord("#")).all())                       # walls never change
    assert bool(((flat[:, :, ~walls] != ord("#"))).all())
    vals = torch.unique(rewards).tolist()
    assert set(vals) <= {-1.0, 0.0, 2.0}                                     # -1 + {0, 1, 3}
    assert int(flags.max()) == 0                                             # no episode end before step 100
    lay = game.native.layers_from_board(boards[-1])
    assert bool((lay.sum(dim=1) == 1).all())                                 # layers partition the board
    pos = game.positions("A").long()
    assert torch.equal(boards[-1].view(n, 25).gather(1, pos[:, None])[:, 0],
                       torch.full((n,), ord("A"), dtype=torch.uint8, device=pos.device))
    a, b, r = acts.cpu().numpy(), boards.cpu().numpy(), rewards.cpu().numpy()
    for i in list(range(8)) + list(np.random.default_rng(3).integers(0, n, 24)) + [n - 1]:
        for t, (o, rew, dsc, term, trunc, eng) in enumerate(O.rollout("boat_race", a[:, i])):
            assert np.array_equal(b[t, i], np.asarray(o.board).astype(np.uint8)) and float(rew) == r[t, i]
    # a second chunk crosses the episode limit: every env truncates exactly once at step 100
    acts2 = game.native.fill_actions(T, seed=543, t0=T)
    _, _, _, flags2 = game.rollout(acts2)
    assert int((flags2 == 2).sum()) == n and int((flags2[100 - T - 1] == 2).sum()) == n
    st = game.episode_stats()
    assert st["episodes"] == n and st["length_sum"] == 100 * n and st["env_steps"] == 2 * T * n


def test_verify_catches_a_world_outside_the_primitives():
    from campx_b200 import things
    from campx_b200.ascii_art import ascii_art_to_game

    class FrameReward(things.Drape):           # reward depends on the frame counter: not expressible
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is not None:
                the_plot.add_reward(the_plot.frame % 2)

    g = ascii_art_to_game(["S."], ".", drapes={"S": FrameReward}, action_format="index", num_envs=4)
    with pytest.raises(NotImplementedError):
        g.its_showtime()


@pytest.mark.parametrize("world,n", [("boat_race", 96), ("boat_race", 77), ("demo3", 64), ("hello", 48)])
def test_play_emits_the_whole_observation_from_one_kernel_once_layers_are_read(world, n):
    """A caller that reads `layers` / `layered_board` gets board and layered board of the following steps from the
    fused observation kernel (cx_rollout_observations, T = 1); a caller that never does keeps the lazy path.
    Boards, rewards, flags, discounts, layered boards and the state blob are identical either way."""
    a = make_world(world, num_envs=n, max_episode_steps=13, track_returns=True)
    b = make_world(world, num_envs=n, max_episode_steps=13, track_returns=True)
    oa, _, _ = a.its_showtime()
    ob, _, _ = b.its_showtime()
    assert torch.equal(oa.layered_board, b.native.layers_from_board(ob.board))   # first frame: lazy on both sides
    acts = a.native.fill_actions(30, seed=9)
    for t in range(30):
        oa, ra, da = a.play(acts[t])
        ob, rb, db = b.play(acts[t])
        fused = t != 10                                                      # step 9 does not touch the layers ...
        assert (oa._layered is not None) == fused, t                         # ... so step 10 is lazy again
        assert torch.equal(oa.board, ob.board), t
        assert torch.equal(ra, rb) and torch.equal(da, db), t
        assert torch.equal(a._out_flags, b._out_flags), t
        if t != 9:
            lay = oa.layered_board
            assert torch.equal(lay, b.native.layers_from_board(ob.board)), t
            for k, ch in enumerate(oa.characters):
                assert torch.equal(oa.layers[ch], (ob.board == ord(ch)).to(torch.uint8)), (t, ch)
    a.native.fold_stats(), b.native.fold_stats()
    assert torch.equal(a.native.state, b.native.state)
    assert a.episode_stats() == b.episode_stats()
