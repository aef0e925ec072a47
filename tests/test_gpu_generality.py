"""GPU parity of the engine-generality row (SURVEY 8(f) row 3): games whose z-order, sprite visibility or
backdrop change during play.  Fixtures in tests/golden/generality_*.json were recorded from the unmodified
reference; here the CUDA path (through the C ABI) is compared with them, with the numpy oracle on random
batched rollouts with time limits and auto reset, and the render state the kernels keep per env (z-order,
visibility bits, backdrop offset) with the oracle's."""
import json
import os

import numpy as np
import pytest
import torch

from campx_b200 import things
from campx_b200.ascii_art import ascii_art_to_game, Partial
from examples.generality_worlds import make_generality_world, Phantom, Drizzle
from oracle import campx_oracle as O

pytestmark = pytest.mark.gpu


def board_str(b):
    return "".join(chr(int(v)) for v in b.reshape(-1).tolist())


def action_for(world, a):
    if world != "scroll":
        return int(a)
    v = [0] * 5
    v[a] = 1
    return torch.FloatTensor(v)


@pytest.mark.parametrize("world", O.GENERALITY_WORLDS)
def test_fused_rollout_matches_reference_fixtures(golden_dir, world):
    """Every recorded episode as one env of a fused cx_rollout: boards, rewards, None-ness, discounts."""
    with open(os.path.join(golden_dir, "generality_" + world + ".json")) as f:
        fx = json.load(f)
    eps = fx["episodes"]
    T = min(len(e["actions"]) for e in eps)
    game = make_generality_world(world, num_envs=len(eps), auto_reset=False)
    obs, _, _ = game.its_showtime()
    assert game.native.info.path == 2 and game.native.info.dynamic_render == 1
    for i, e in enumerate(eps):
        assert board_str(obs.board[i].cpu()) == e["frames"][0]["board"]
    acts = torch.tensor([e["actions"][:T] for e in eps], dtype=torch.uint8).t().contiguous().cuda()
    boards, rewards, discounts, flags = game.rollout(acts)
    b, r, f = boards.cpu(), rewards.cpu().numpy(), flags.cpu().numpy()
    for i, e in enumerate(eps):
        for t in range(T):
            want = e["frames"][t + 1]
            assert board_str(b[t, i]) == want["board"], (world, e["name"], t)
            assert (want["reward"] is None) == bool(f[t, i] & 4)
            if want["reward"] is not None:
                assert float(r[t, i]) == want["reward"]
            assert want["discount"] == (1.0 if discounts is None else float(discounts[t, i]))


@pytest.mark.parametrize("world", O.GENERALITY_WORLDS)
def test_render_state_matches_oracle(world):
    """cx_get_render_state: the per-env z-order / visibility / backdrop offset equal the oracle's things order,
    Sprite.visible and Backdrop.curtain after every step."""
    n, T = 24, 30
    game = make_generality_world(world, num_envs=n)
    game.its_showtime()
    rng = np.random.Generator(np.random.PCG64(17))
    acts = rng.integers(0, 5, size=(T, n)).astype(np.uint8)
    worlds = [O.World(world) for _ in range(n)]
    ids = "".join(e.character for e in game.spec.entities)          # entity id = initial z index
    base_backdrop = np.asarray(worlds[0].engine.backdrop.curtain).copy()
    for t in range(T):
        game.play(torch.from_numpy(acts[t]).cuda())
        z, vis, off = game.native.render_state()
        z, vis, off = z.cpu().numpy(), vis.cpu().numpy(), off.cpu().numpy()
        for i in range(n):
            worlds[i].step(int(acts[t, i]))
            eng = worlds[i].engine
            got_order = "".join(ids[(int(z[i]) >> (4 * p)) & 15] for p in range(len(ids)))
            assert got_order == "".join(eng.things.keys()), (world, i, t)
            for k, ch in enumerate(ids):
                ent = eng.things[ch]
                if isinstance(ent, O.Sprite):
                    assert bool((int(vis[i]) >> k) & 1) == bool(ent.visible)
            if world == "scroll":
                dr, dc = int(off[i]) // game.cols, int(off[i]) % game.cols
                assert np.array_equal(np.roll(base_backdrop, (dr, dc), axis=(0, 1)), np.asarray(eng.backdrop.curtain))


def test_hidden_sprite_behind_the_first_drape_stops_stamping():
    """Quirk Q1 meets visibility: a sprite behind the first drape stamps the backdrop only while visible; the
    stamps it left stay.  Four phantoms, two of which start hidden, 13x9 board (generic kernel, ragged batch)."""
    art = ['G...@....',
           '....@....',
           'H...@...J',
           '.........',
           '..@@@....',
           '.........',
           'K........',
           '.........',
           '.........',
           '.........',
           '.........',
           '.........',
           '........#']
    n, T = 37, 60

    def user():
        return ascii_art_to_game(art, '.',
                                 sprites={'G': Partial(Phantom, True, 1, 1, True), 'H': Partial(Phantom, False, 1, -1, False),
                                          'J': Partial(Phantom, False, -1, 1, True), 'K': Partial(Phantom, True, -1, -1, False)},
                                 drapes={'@': Drizzle, '#': things.FixedDrape},
                                 update_schedule='GHJK@#', z_order='GH@JK#', num_envs=n)

    def oracle():
        ghost = lambda vis, dr, dc, sw: (O.GhostSprite, (vis, dr, dc), dict(switchable=sw))
        return O.ascii_art_to_game(art, '.',
                                   sprites={'G': ghost(True, 1, 1, True), 'H': ghost(False, 1, -1, False),
                                            'J': ghost(False, -1, 1, True), 'K': ghost(True, -1, -1, False)},
                                   drapes={'@': O.RainDrape, '#': O.FixedDrape},
                                   update_schedule='GHJK@#', z_order='GH@JK#')

    game = user()
    game.its_showtime()
    assert game.native.info.has_dynamic_backdrop == 1
    oracles = [oracle() for _ in range(n)]
    for o in oracles:
        o.its_showtime()
    rng = np.random.Generator(np.random.PCG64(4))
    acts = rng.integers(0, 5, size=(T, n)).astype(np.uint8)
    boards, rewards, _, flags = game.rollout(torch.from_numpy(acts).cuda())
    b = boards.cpu().numpy()
    for i in range(n):
        for t in range(T):
            o, rew, dsc = oracles[i].play(int(acts[t, i]))
            assert np.array_equal(b[t, i], np.asarray(o.board).astype(np.uint8)), (i, t)
            assert float(rew) == float(rewards[t, i])
    assert (b == ord('J')).any() and (b == ord('H')).any()


@pytest.mark.parametrize("world", O.GOAL_WORLDS)
@pytest.mark.parametrize("route", ["auto", "wt64", "wt128", "obs", "stg", "tiles_for_single_steps"])
def test_reach_the_goal_worlds(golden_dir, world, route, monkeypatch):
    """terminate_episode that depends on the cell the agent reached (ADVICE r1): reference-recorded episodes as envs
    of a fused rollout, then random rollouts with auto reset against the oracle, step-by-step play() included.
    `goal` is a single-agent game (transition table with per-cell termination and discount, every kernel build),
    `goal2` runs on the generic kernels (directives replayed per step in update order)."""
    if route != "auto":
        monkeypatch.setenv("CX_ROUTE", {"wt64": "tile64", "wt128": "tile128", "obs": "obs", "stg": "lane",
                                        "tiles_for_single_steps": "no_step_composer"}[route])
    with open(os.path.join(golden_dir, "generality_" + world + ".json")) as f:
        eps = json.load(f)["episodes"]
    T = max(len(e["actions"]) for e in eps)
    game = make_generality_world(world, num_envs=len(eps), auto_reset=False)
    game.its_showtime()
    assert game.native.info.path == (1 if world == "goal" else 2) and game.native.can_terminate
    acts = torch.tensor([(e["actions"] + [4] * T)[:T] for e in eps], dtype=torch.uint8).t().contiguous().cuda()
    boards, rewards, discounts, flags = game.rollout(acts)
    b, r, d, f = boards.cpu(), rewards.cpu().numpy(), discounts.cpu().numpy(), flags.cpu().numpy()
    for i, e in enumerate(eps):
        for t in range(len(e["actions"])):
            want = e["frames"][t + 1]
            assert board_str(b[t, i]) == want["board"], (world, e["name"], t)
            assert float(r[t, i]) == want["reward"] and float(d[t, i]) == want["discount"], (world, e["name"], t)
            assert bool(f[t, i] & 1) == (e["error_after"] is not None and t == len(e["actions"]) - 1)
        if e["error_after"]:                                   # frozen afterwards (auto_reset = False)
            assert all(int(f[t, i]) & 8 for t in range(len(e["actions"]), T))
    # random rollouts, auto reset + time limit, fused and step by step, against the oracle rebuilt at every end
    n, T, limit = 96, 50, 17
    game = make_generality_world(world, num_envs=n, max_episode_steps=limit, track_returns=True)
    step = make_generality_world(world, num_envs=n, max_episode_steps=limit, track_returns=True)
    game.its_showtime()
    step.its_showtime()
    acts = game.native.fill_actions(T, seed=31)
    boards, rewards, discounts, flags = game.rollout(acts)
    for t in range(T):
        obs, rew, dsc = step.play(acts[t])
        assert torch.equal(obs.board, boards[t]) and torch.equal(rew, rewards[t]) and torch.equal(dsc, discounts[t])
        assert torch.equal(step.flags, flags[t])
    a, b = acts.cpu().numpy(), boards.cpu().numpy()
    r, d, f = rewards.cpu().numpy(), discounts.cpu().numpy(), flags.cpu().numpy()
    ended = 0
    for i in list(range(0, n, 7)) + [n - 1]:
        for t, (o, rew, dsc, term, trunc, eng) in enumerate(
                O.rollout(world, a[:, i], rebuild_on_done=True, max_episode_steps=limit)):
            assert np.array_equal(b[t, i], np.asarray(o.board).astype(np.uint8)), (world, i, t)
            assert float(rew) == float(r[t, i]) and float(dsc) == float(d[t, i]), (world, i, t)
            assert term == bool(f[t, i] & 1) and trunc == bool(f[t, i] & 2), (world, i, t)
            ended += term
    assert ended > 0


def test_unsupported_combination_is_refused():
    """A rolling backdrop together with backdrop-stamping sprites is outside the primitives: refused loudly."""
    from examples.generality_worlds import Panorama, Climber

    class IntPanorama(Panorama):
        def update(self, actions, board, layers, all_things, the_plot):
            if actions is None:
                return
            v = [0] * 5
            v[int(actions)] = 1
            super().update(v, board, layers, all_things, the_plot)

    g = ascii_art_to_game(['S.~', '.W.'], '.', sprites={'S': Climber}, drapes={'W': things.FixedDrape},
                          backdrop=IntPanorama, z_order='SW', update_schedule='SW', num_envs=8)
    with pytest.raises(NotImplementedError):
        g.its_showtime()
