"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.json from the UNMODIFIED reference.

Run against a checkout of the original CampX:

    CAMPX_REFERENCE_ROOT=<checkout> python oracle/gen_golden.py

The reference (`campx/` + `examples/boat_race.py` of that checkout + the game-defining cells of the
Demo 1-4 / Hello World notebooks) is executed under `oracle/shim.py`; nothing is copied from it.
Each fixture holds action sequences and, per frame, the board, every layer, entity state, the
backdrop curtain (pins quirk Q1), reward (value and None-ness) and discount.  Action streams are
drawn from numpy's PCG64 with the seed stored in the fixture, so they can be re-derived.

The fixtures are small (a few hundred kB in total) and committed, so the tests check the CUDA path
and the numpy oracle against them without the checkout.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import shim  # noqa: E402

shim.install()

import torch  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
REF_COMMIT = "90248b4"


def ref_frame_record(game, obs, reward, discount):
    from campx import things as ref_things
    things = {}
    for ch, ent in game._sprites_and_drapes.items():
        if isinstance(ent, ref_things.Sprite):
            things[ch] = {"pos": [int(ent.position[0]), int(ent.position[1])],
                          "visible": bool(ent.visible)}
        else:
            things[ch] = {"mask": "".join(str(int(v)) for v in ent.curtain.reshape(-1).tolist())}
    return {
        "board": "".join(chr(int(v)) for v in obs.board.reshape(-1).tolist()),
        "layers": {ch: "".join(str(int(v)) for v in l.reshape(-1).tolist())
                   for ch, l in sorted(obs.layers.items())},
        "reward": None if reward is None else float(reward),
        "reward_type": type(reward).__name__ if not torch.is_tensor(reward) else str(reward.dtype),
        "discount": float(discount),
        "things": things,
        "backdrop": "".join(chr(int(v)) for v in game._backdrop.curtain.reshape(-1).tolist()),
        "z_order": "".join(game._sprites_and_drapes.keys()),
    }


def encode_action(world, index):
    if world in ("hello", "zswap", "ghost"):
        return int(index)
    onehot = [0] * 5
    onehot[int(index)] = 1
    if world in ("boat_race", "demo4", "scroll", "goal", "goal2"):
        return torch.FloatTensor(onehot)
    return onehot


_NOTEBOOKS = {
    "demo1": "Demo 1: Simple Agent Example.ipynb",
    "demo2": "Demo 2: Simple Wall Example.ipynb",
    "demo3": "Demo 3: Hover Reward Example.ipynb",
    "demo4": "Demo 4: Directional Hover Reward Example.ipynb",
    "hello": "Hello World Example.ipynb",
}
_ns_cache = {}


# ---- engine-generality worlds (SURVEY 8(f) row 3), written against the REFERENCE API -------------------------
# None of the reference's own worlds changes its z-order, hides a sprite or updates its backdrop, so these
# three small worlds exercise campx/engine.py:242-281,163 (z-order directives + re-render), things.py:320,
# 390-392 + engine.py:315 (Sprite.visible) and things.py:103-148 (Backdrop.update) on the reference itself.
ZSWAP_ART = ["S.....",
             ".XX.Y.",
             ".XXYY.",
             "...YY.",
             "......"]
GHOST_ART = ["G..@.",
             "..@..",
             "H...."]
SCROLL_ART = ["A.~~.^",
              ".~..^.",
              "~..^..",
              "..^..~"]
GOAL_ART = ["######", "#A  G#", "# #  #", "#   X#", "######"]
GOAL2_ART = ["######", "#A  G#", "# #  #", "#S  X#", "######"]
GENERALITY_WORLDS = ("zswap", "ghost", "scroll", "goal", "goal2")


def make_ref_generality_game(world):
    from campx import things
    from campx.ascii_art import ascii_art_to_game, Partial

    def roll(t, shift, axis):
        return torch.from_numpy(np.roll(t.numpy(), shift, axis).copy())

    if world == "zswap":
        class XDrape(things.Drape):
            def update(self, actions, board, layers, backdrop, all_things, the_plot):
                if actions is None:
                    return
                if actions == 0:
                    self.curtain.set_(roll(self.curtain, 1, 1))
                    the_plot.add_reward(1)
                if actions == 1:
                    the_plot.change_z_order("X", "Y")
                if actions == 2:
                    the_plot.change_z_order("Y", None)
                if actions == 3:
                    the_plot.change_z_order("X", None)
                    the_plot.change_z_order("Y", "X")

        class SSprite(things.Sprite):
            def update(self, actions, board, layers, backdrop, all_things, the_plot):
                if actions is None:
                    return
                row, col = self.position
                if actions == 0:
                    col = (col + 1) % self.corner.col
                if actions == 1:
                    row = (row + 1) % self.corner.row
                self._position = self.Position(row, col)
                if actions == 4:
                    the_plot.change_z_order("S", "Y")
                if actions == 2:
                    the_plot.change_z_order("S", None)

        return ascii_art_to_game(ZSWAP_ART, ".", sprites={"S": SSprite},
                                 drapes={"X": XDrape, "Y": things.FixedDrape},
                                 update_schedule="SXY", z_order="SXY")
    if world == "ghost":
        class Ghost(things.Sprite):
            def __init__(self, corner, position, character, start_visible, d_row, d_col):
                super(Ghost, self).__init__(corner, position, character)
                self._visible = start_visible
                self._d = (d_row, d_col)

            def update(self, actions, board, layers, backdrop, all_things, the_plot):
                if actions is None:
                    return
                row, col = self.position
                if actions == 0:
                    col = (col + self._d[1]) % self.corner.col
                if actions == 1:
                    row = (row + self._d[0]) % self.corner.row
                self._position = self.Position(row, col)
                if self.character == "G":
                    if actions == 2:
                        self._visible = False
                    if actions == 3:
                        self._visible = True
                if actions == 4:
                    self._visible = not self._visible

        class Rain(things.Drape):
            def update(self, actions, board, layers, backdrop, all_things, the_plot):
                if actions is None:
                    return
                if actions == 1:
                    self.curtain.set_(roll(self.curtain, 1, 0))
                the_plot.add_reward(0.5)

        return ascii_art_to_game(GHOST_ART, ".",
                                 sprites={"G": Partial(Ghost, True, 1, 1), "H": Partial(Ghost, False, 1, -1)},
                                 drapes={"@": Rain}, update_schedule="GH@", z_order="GH@")
    if world in ("goal", "goal2"):
        # "reach the goal": a tile watches the agent (like boat_race.py:79-82) and calls terminate_episode
        # (plot.py:161-184) when the agent stands on it
        import boat_race

        class Seeker(boat_race.AgentDrape):       # the reference's own agent, walls '#'
            def update(self, actions, board, layers, backdrop, all_things, the_plot):
                super(Seeker, self).update(actions, board, layers, backdrop, all_things, the_plot)
                if actions is not None:
                    the_plot.add_reward(-1)

        class Exit(things.Drape):
            def __init__(self, curtain, character, prize, pcontinue=0.0):
                super(Exit, self).__init__(curtain, character)
                self.prize, self.pcontinue = prize, pcontinue

            def update(self, actions, board, layers, backdrop, all_things, the_plot):
                if actions is None:
                    return
                here = (all_things["A"].curtain * layers[self.character]).sum()
                the_plot.add_reward(here * self.prize)
                if here > 0:
                    the_plot.terminate_episode(self.pcontinue)

        class Drifter(things.Sprite):
            def update(self, actions, board, layers, backdrop, all_things, the_plot):
                if actions is None:
                    return
                self._position = self.Position(self.position.row, (self.position.col + 1) % self.corner.col)

        drapes = {"A": Seeker, "#": things.FixedDrape, "G": Partial(Exit, 10), "X": Partial(Exit, -5, 0.25)}
        if world == "goal":
            return ascii_art_to_game(GOAL_ART, " ", drapes=drapes, update_schedule="AGX#", z_order="GXA#")
        return ascii_art_to_game(GOAL2_ART, " ", sprites={"S": Drifter}, drapes=drapes,
                                 update_schedule="ASGX#", z_order="GXAS#")
    if world == "scroll":
        import boat_race

        class Scroller(things.Backdrop):
            def update(self, actions, board, layers, all_things, the_plot):
                if actions is None:
                    return
                a = int(torch.as_tensor(actions).argmax())
                if a < 4:
                    shift, axis = ((-1, 1), (1, 1), (-1, 0), (1, 0))[a]
                    self.curtain.set_(roll(self.curtain, shift, axis))

        class Hiker(boat_race.AgentDrape):       # the reference's own agent: stops at '^' instead of '#'
            def update(self, actions, board, layers, backdrop, all_things, the_plot):
                super(Hiker, self).update(actions, board, layers, backdrop, all_things, the_plot)
                if actions is not None:
                    the_plot.add_reward(1)

        return ascii_art_to_game(SCROLL_ART, ".", drapes={"A": Partial(Hiker, blocking_chars="^")},
                                 backdrop=Scroller, z_order="A")
    raise KeyError(world)


def make_ref_game(world):
    """-> (game, first_obs, first_reward, first_discount) from the reference's own make_game()."""
    if world in GENERALITY_WORLDS:
        game = make_ref_generality_game(world)
        obs, reward, discount = game.its_showtime()
        return game, obs, reward, discount
    if world == "boat_race":
        import boat_race
        return boat_race.make_game()
    if world not in _ns_cache:
        _ns_cache[world] = shim.load_notebook_world(_NOTEBOOKS[world])
    out = _ns_cache[world]["make_game"]()
    if isinstance(out, tuple):          # Demo 4's make_game already calls its_showtime
        return out
    obs, reward, discount = out.its_showtime()
    return out, obs, reward, discount


def run_episode(world, actions, expect_error_after_end=True):
    game, obs, reward, discount = make_ref_game(world)
    frames = [ref_frame_record(game, obs, reward, discount)]
    played = []
    error = None
    for a in actions:
        try:
            obs, reward, discount = game.play(encode_action(world, a))
        except RuntimeError as e:       # play() after game over (engine.py:149-151)
            error = str(e)
            break
        played.append(int(a))
        frames.append(ref_frame_record(game, obs, reward, discount))
    return {"actions": played, "frames": frames, "error_after": error,
            "rows": game._rows, "cols": game._cols}


def world_fixture(world, scripted, n_random, random_len, seed, action_hi):
    episodes = []
    for name, acts in scripted:
        ep = run_episode(world, acts)
        ep["name"] = name
        episodes.append(ep)
    rng = np.random.Generator(np.random.PCG64(seed))
    for i in range(n_random):
        acts = rng.integers(0, action_hi, size=random_len).tolist()
        ep = run_episode(world, acts)
        ep["name"] = "random_%d" % i
        episodes.append(ep)
    return {"world": world, "source": "reference@%s executed under oracle/shim.py" % REF_COMMIT,
            "generator": "oracle/gen_golden.py", "seed": seed, "episodes": episodes}


def engine_semantics_fixture():
    """Small custom worlds against the reference API pinning SURVEY Appendix A.7 behaviours."""
    from campx import things
    from campx.ascii_art import ascii_art_to_game

    cases = {}

    class TwoRewards(things.Drape):
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is None:
                return
            the_plot.add_reward(1)
            the_plot.add_reward(2.5)
            if actions == 2:
                the_plot.change_default_discount(0.5)
            if actions == 3:
                the_plot.terminate_episode()

    game = ascii_art_to_game(["X.", ".."], ".", drapes={"X": TwoRewards})
    game.its_showtime()
    seq = []
    for a in (0, 2, 0, 3):
        _, r, d = game.play(a)
        seq.append({"action": a, "reward": float(r), "discount": float(d)})
    try:
        game.play(0)
        seq.append({"error": None})
    except RuntimeError as e:
        seq.append({"error": str(e)})
    cases["reward_sum_discount_terminate"] = seq

    # update groups: W copies where M *appears in layers*; with [['M'],['W']] it sees M's move in
    # the same step (re-render between groups, engine.py:195-208), with a flat schedule it lags.
    class Mover(things.Drape):
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is None:
                return
            b = self.curtain
            self.curtain.set_(torch.cat([b[:, -1:], b[:, :-1]], dim=1))

    class Watcher(things.Drape):
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is None:
                return
            the_plot.add_reward(int((layers["M"][0] * torch.arange(4).byte()).sum()))

    for label, sched in (("grouped", [["M"], ["W"]]), ("flat", ["M", "W"])):
        game = ascii_art_to_game(["M...", "W..."], ".", drapes={"M": Mover, "W": Watcher},
                                 update_schedule=sched, z_order="MW")
        game.its_showtime()
        rs = []
        for _ in range(3):
            _, r, _ = game.play(0)
            rs.append(float(r))
        cases["update_groups_" + label] = rs

    class Swapper(things.Drape):
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions == 1:
                the_plot.change_z_order("X", "Y")
            if actions == 2:
                the_plot.change_z_order("Y", None)

    game = ascii_art_to_game(["X"], ".", drapes={"X": Swapper, "Y": things.FixedDrape},
                             update_schedule="XY", z_order="XY")
    # Y has an empty mask in the art; give it the same cell so occlusion is observable
    game._sprites_and_drapes["Y"].curtain.fill_(1)
    obs, _, _ = game.its_showtime()
    zs = [{"z": "".join(game._sprites_and_drapes.keys()), "board": int(obs.board[0, 0])}]
    for a in (0, 1, 0, 2):
        obs, _, _ = game.play(a)
        zs.append({"action": a, "z": "".join(game._sprites_and_drapes.keys()),
                   "board": int(obs.board[0, 0])})
    cases["change_z_order"] = zs

    # a world with sprites but no drape: quirk Q1(ii), the backdrop is zeroed at every render
    class Still(things.Sprite):
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is None:
                return
            self._position = self.Position(self._position.row, (self._position.col + 1) % self.corner.col)

    game = ascii_art_to_game(["P..", "..."], ".", sprites={"P": Still})
    obs, _, _ = game.its_showtime()
    boards = [[int(v) for v in obs.board.reshape(-1).tolist()]]
    for _ in range(2):
        obs, _, _ = game.play(0)
        boards.append([int(v) for v in obs.board.reshape(-1).tolist()])
    cases["sprite_only_world_boards"] = boards
    return {"world": "engine_semantics", "source": "reference@%s executed under oracle/shim.py" % REF_COMMIT,
            "generator": "oracle/gen_golden.py", "cases": cases}


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    preset = [1, 1, 3, 3, 0, 0, 2, 2, 3, 3, 1, 1, 2, 2, 0, 0, 0, 4, 4, 4]   # select_action_preset(t), boat_race.py:154-184
    import boat_race
    assert preset == [int(boat_race.select_action_preset(t).argmax()) for t in range(20)]
    jobs = {
        "boat_race": dict(scripted=[("preset_lap", preset)], n_random=4, random_len=120, seed=543, action_hi=5),
        "demo1": dict(scripted=[("notebook", [0]), ("survey_a2", [0, 0, 2, 2, 3, 4, 1])],
                      n_random=2, random_len=80, seed=11, action_hi=5),
        "demo2": dict(scripted=[("notebook", [1, 1, 1]), ("survey_a3", [1, 1, 1, 3, 3, 0, 2, 4])],
                      n_random=2, random_len=80, seed=12, action_hi=5),
        "demo3": dict(scripted=[("notebook", [1]), ("survey_a4", [1, 4, 1, 0, 3, 2, 0, 3, 3])],
                      n_random=2, random_len=80, seed=13, action_hi=5),
        "demo4": dict(scripted=[("notebook", [1, 3, 0, 2]), ("survey_a5", [1, 3, 0, 2, 1, 1, 3, 0, 1, 3])],
                      n_random=2, random_len=80, seed=14, action_hi=5),
        "hello": dict(scripted=[("notebook_up3_quit", [0, 0, 0, 4, 0]),
                                ("each_action", [0, 1, 2, 3, 3, 2, 1, 0, 4])],
                      n_random=2, random_len=30, seed=15, action_hi=4),
    }
    for world, kw in jobs.items():
        fx = world_fixture(world, **kw)
        path = os.path.join(GOLDEN_DIR, world + ".json")
        with open(path, "w") as f:
            json.dump(fx, f, separators=(",", ":"))
        print(world, "->", path, os.path.getsize(path), "bytes;",
              sum(len(e["frames"]) for e in fx["episodes"]), "frames")
    gen_jobs = {
        "zswap": dict(scripted=[("each_action", [0, 1, 0, 2, 0, 3, 4, 0, 1, 2, 1, 1, 0, 3, 0, 0, 4])],
                      n_random=3, random_len=60, seed=21, action_hi=5),
        "ghost": dict(scripted=[("each_action", [0, 1, 2, 0, 3, 4, 1, 4, 0, 0, 2, 2, 3, 1, 4, 4])],
                      n_random=3, random_len=60, seed=22, action_hi=5),
        "scroll": dict(scripted=[("each_action", [0, 1, 1, 2, 3, 3, 4, 1, 1, 1, 3, 0, 2, 2])],
                       n_random=3, random_len=60, seed=23, action_hi=5),
    }
    # paths to the exit (3 x right) and to the pit (down, down, right x 3), then random walks that end early
    gen_jobs["goal"] = dict(scripted=[("to_exit", [1, 1, 1, 4]), ("to_pit", [3, 3, 1, 1, 1, 4]), ("bump", [0, 2, 4, 1, 3, 3])],
                            n_random=6, random_len=40, seed=24, action_hi=5)
    gen_jobs["goal2"] = dict(scripted=[("to_exit", [1, 1, 1, 4]), ("to_pit", [3, 3, 1, 1, 1, 4])],
                             n_random=6, random_len=40, seed=25, action_hi=5)
    for world, kw in gen_jobs.items():
        fx = world_fixture(world, **kw)
        path = os.path.join(GOLDEN_DIR, "generality_" + world + ".json")
        with open(path, "w") as f:
            json.dump(fx, f, separators=(",", ":"))
        print(world, "->", path, os.path.getsize(path), "bytes;",
              sum(len(e["frames"]) for e in fx["episodes"]), "frames")
    fx = engine_semantics_fixture()
    path = os.path.join(GOLDEN_DIR, "engine_semantics.json")
    with open(path, "w") as f:
        json.dump(fx, f, indent=1)
    print("engine_semantics ->", path)
    print(json.dumps(fx["cases"], indent=1)[:1500])


if __name__ == "__main__":
    main()
