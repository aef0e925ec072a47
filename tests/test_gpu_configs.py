"""BASELINE.json configs [1] and [2] at their stated sizes, through the public API:

  [1] Hello World / Demo 1, 65,536 batched envs on one B200
  [2] Demo 2 (wall) + Demo 4 (directional hover reward), 2^20 batched envs, bit-exact vs the reference

At these sizes the oracle cannot replay every env, so each test checks size-independent properties of the
whole batch on the device (entity counts per board, static scenery, reward alphabet, flag/action
consistency, layers partition the board, episode statistics) and replays a sample of envs -- the first
ones, the last one and random ones -- through the oracle for exact equality of board, reward and flags.
"""
import numpy as np
import pytest
import torch

from campx_b200 import _native as N
from examples.worlds import make_world
from oracle import campx_oracle as O

pytestmark = pytest.mark.gpu


def sample_envs(n, k, seed):
    return list(range(4)) + [int(i) for i in np.random.default_rng(seed).integers(0, n, k)] + [n - 1]


def replay(world, acts, boards, rewards, flags, envs, limit):
    a, b, r, f = acts.cpu().numpy(), boards.cpu().numpy(), rewards.cpu().numpy(), flags.cpu().numpy()
    for i in envs:
        for t, (o, rew, dsc, term, trunc, eng) in enumerate(
                O.rollout(world, a[:, i], rebuild_on_done=True, max_episode_steps=limit)):
            assert np.array_equal(b[t, i], np.asarray(o.board).astype(np.uint8)), (world, i, t)
            assert (0.0 if rew is None else float(rew)) == float(r[t, i]), (world, i, t)
            assert term == bool(f[t, i] & N.CX_FLAG_TERMINATED) and trunc == bool(f[t, i] & N.CX_FLAG_TRUNCATED)
            assert (rew is None) == bool(f[t, i] & N.CX_FLAG_REWARD_NONE)


def test_config1_demo1_65536_envs():
    n, T, limit = 65536, 48, 40
    game = make_world("demo1", num_envs=n, max_episode_steps=limit, track_returns=True)
    game.its_showtime()
    acts = game.native.fill_actions(T, seed=11)
    boards, rewards, discounts, flags = game.rollout(acts)
    flat = boards.view(T, n, 25)
    agents = (flat == ord("A")).sum(dim=2)
    assert int(agents.min()) == 1 and int(agents.max()) == 1           # the agent never vanishes (toroidal, Q5)
    assert bool((rewards == 1.0).all())                                  # Demo 1 pays 1 every step
    assert int((flags == N.CX_FLAG_TRUNCATED).sum()) == n                # one time-limit hit per env in 48 steps
    assert int((flags[limit - 1] == N.CX_FLAG_TRUNCATED).sum()) == n
    art = torch.tensor([ord(c) for c in "".join(O.DEMO_ART).replace("A", " ")], dtype=torch.uint8, device=flat.device)
    not_agent = flat != ord("A")
    assert bool((flat[not_agent] == art.expand(T, n, 25)[not_agent]).all())   # scenery under the agent only
    lay = game.native.layers_from_board(boards[-1])
    assert bool((lay.sum(dim=1) == 1).all())
    st = game.episode_stats()
    assert st["episodes"] == n and st["return_sum"] == float(limit) * n and st["env_steps"] == n * T
    replay("demo1", acts, boards, rewards, flags, sample_envs(n, 20, 1), limit)


def test_config1_hello_world_65536_envs():
    n, T, limit = 65536, 24, 20
    game = make_world("hello", num_envs=n, max_episode_steps=limit, track_returns=True)
    game.its_showtime()
    acts = game.native.fill_actions(T, seed=12)                          # uniform over 0..4
    keep_quit = torch.rand(acts.shape, device=acts.device) < 0.1         # ~2% quit (action 4)
    acts = torch.where((acts == 4) & ~keep_quit, acts % 3, acts).contiguous()
    boards, rewards, discounts, flags = game.rollout(acts)
    flat = boards.view(T, n, -1)
    cells = flat.shape[2]
    assert cells == 13 * 36
    top = (flat == ord("4")).sum(dim=2)                                  # the front-most sprite is always visible
    assert int(top.min()) == 1 and int(top.max()) == 1
    assert int((flat == ord("3")).sum(dim=2).max()) == 1                 # '3' only hides behind '4'
    at = (flat == ord("@")).sum(dim=2)                                   # 59 cells minus those under '3' / '4'
    assert int(at.max()) <= 59 and int(at.min()) >= 57
    quit_ = acts == 4
    term = (flags & N.CX_FLAG_TERMINATED) != 0
    assert torch.equal(term, quit_)                                      # terminate_episode() iff action 4
    assert torch.equal((flags & N.CX_FLAG_REWARD_NONE) != 0, quit_)      # ... and then nobody adds a reward
    assert bool((rewards[~quit_] == 1.0).all()) and bool((rewards[quit_] == 0.0).all())
    assert bool((discounts[quit_] == 0.0).all()) and bool((discounts[~quit_] == 1.0).all())
    known = torch.zeros(256, dtype=torch.bool, device=flat.device)
    known[[ord(c) for c in "1234@# "]] = True
    for t in range(T):
        assert bool(known[flat[t].long()].all())                         # nothing but game characters on the board
    lay = game.native.layers_from_board(boards[-1])
    assert bool((lay.sum(dim=1) == 1).all())
    st = game.episode_stats()
    ended = int(((flags & (N.CX_FLAG_TERMINATED | N.CX_FLAG_TRUNCATED)) != 0).sum())
    assert st["episodes"] == ended and st["env_steps"] == n * T
    replay("hello", acts, boards, rewards, flags, sample_envs(n, 10, 2), limit)


@pytest.mark.parametrize("world", ["demo2", "demo4"])
def test_config2_walls_and_hover_rewards_2pow20_envs(world):
    n, T, limit = 1 << 20, 32, 25
    game = make_world(world, num_envs=n, max_episode_steps=limit, track_returns=True)
    game.its_showtime()
    acts = game.native.fill_actions(T, seed=21)
    boards, rewards, discounts, flags = game.rollout(acts)
    flat = boards.view(T, n, 25)
    agents = (flat == ord("A")).sum(dim=2)
    assert int(agents.min()) == 1 and int(agents.max()) == 1
    art = "".join(O.DEMO_ART if world == "demo2" else O.BOAT_RACE_ART)
    walls = torch.tensor([c == "#" for c in art], device=flat.device)
    assert bool((flat[:, :, walls] == ord("#")).all())                   # the agent never enters a wall
    assert bool((flat[:, :, ~walls] != ord("#")).all())
    vals = set(torch.unique(rewards).tolist())
    assert vals == ({1.0} if world == "demo2" else {0.0, 1.0})           # Demo 2: 1 per step; Demo 4: hover 0/1
    assert int((flags == N.CX_FLAG_TRUNCATED).sum()) == n and int((flags[limit - 1] == N.CX_FLAG_TRUNCATED).sum()) == n
    lay = game.native.layers_from_board(boards[-1])
    assert bool((lay.sum(dim=1) == 1).all())
    st = game.episode_stats()
    assert st["episodes"] == n and st["env_steps"] == n * T
    if world == "demo2":
        assert st["return_sum"] == float(limit) * n
    # fused rollout == the same steps played one at a time (first 3 steps, whole batch)
    game2 = make_world(world, num_envs=n, max_episode_steps=limit, track_returns=True)
    game2.its_showtime()
    for t in range(3):
        obs, rew, _ = game2.play(acts[t])
        assert torch.equal(obs.board.view(n, 25), flat[t]) and torch.equal(rew, rewards[t])
    replay(world, acts, boards, rewards, flags, sample_envs(n, 24, 3), limit)


@pytest.mark.parametrize("n", [49152, 57344 + 16 * 37])
def test_one_wave_build_matches_the_standard_build(n):
    """Batches that need 21..28 warps per SM run on the fat-CTA build of the register-state kernel (two CTAs of up to 14
    warps per SM, one wave; cx_launch_generic_rollout).  Environments are independent, so any 64 of them replayed in a
    64-env batch (standard build) must give the same boards, rewards, flags and discounts."""
    T = 14
    big = make_world("hello", num_envs=n, max_episode_steps=9, track_returns=True, verify=False)
    small = make_world("hello", num_envs=64, max_episode_steps=9, track_returns=True, verify=False)
    big.its_showtime()
    small.its_showtime()
    acts = big.native.fill_actions(T, seed=77)
    boards, rewards, discounts, flags = big.rollout(acts)
    pick = torch.cat([torch.arange(0, 16), torch.arange(n // 2 - 16, n // 2 + 16), torch.arange(n - 16, n)]).cuda()
    b2, r2, d2, f2 = small.rollout(acts[:, pick].contiguous())
    assert torch.equal(boards[:, pick], b2) and torch.equal(rewards[:, pick], r2) and torch.equal(flags[:, pick], f2)
    assert (discounts is None and d2 is None) or torch.equal(discounts[:, pick], d2)
    assert big.episode_stats()["env_steps"] == n * T


def test_register_state_kernel_builds_agree(monkeypatch):
    """The three builds of the register-state generic kernel (5 CTAs x 96 registers, 6 x 80, two fat CTAs x 72) are the
    same source under different launch bounds; cx_launch_generic_rollout picks one by batch size.  Forced through
    CX_ROUTE=gen96 / gen80 / gen_wave they must produce identical rollouts and final states."""
    n, T = 1024, 40
    results = []
    for build in ("gen96", "gen80", "gen_wave"):
        monkeypatch.setenv("CX_ROUTE", build)
        game = make_world("hello", num_envs=n, max_episode_steps=11, track_returns=True, verify=False)
        game.its_showtime()
        acts = game.native.fill_actions(T, seed=5)
        boards, rewards, discounts, flags = game.rollout(acts)
        game.native.fold_stats()   # partial statistics blocks follow the launch geometry
        results.append((boards.clone(), rewards.clone(), flags.clone(), game.native.state.clone(), game.episode_stats()))
    monkeypatch.delenv("CX_ROUTE")
    for other in results[1:]:
        for x, y in zip(results[0][:4], other[:4]):
            assert torch.equal(x, y)
        assert results[0][4] == other[4]
    # and the first of them against the oracle on a few envs
    replay("hello", acts, results[0][0], results[0][1], results[0][2], [0, 1, 511, n - 1], 11)
