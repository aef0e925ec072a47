"""Pins oracle/campx_oracle.py (numpy restatement) to the reference.

1. against the committed fixtures in tests/golden/ (made by oracle/gen_golden.py from the unmodified
   reference under oracle/shim.py) -- runs everywhere, including the GPU box;
2. against the reference executed live, when CAMPX_REFERENCE_ROOT names a checkout of it.
"""
import json
import os

import numpy as np
import pytest

from oracle import campx_oracle as O
from oracle import shim

# the six reference worlds + the three engine-generality worlds (SURVEY 8(f) row 3: z-order directives, sprite
# visibility, scrolling backdrop), all recorded from the reference itself by oracle/gen_golden.py
# + two "reach the goal" worlds whose terminate_episode depends on where the agent stands
WORLDS = ["boat_race", "demo1", "demo2", "demo3", "demo4", "hello", "zswap", "ghost", "scroll", "goal", "goal2"]


def load(golden_dir, world):
    name = ("generality_" + world) if world in O.GENERALITY_WORLDS + O.GOAL_WORLDS else world
    with open(os.path.join(golden_dir, name + ".json")) as f:
        return json.load(f)


def assert_frame_equal(got, want, ctx):
    for key in ("board", "layers", "things", "backdrop", "z_order"):
        assert got[key] == want[key], "%s: %s differs\n got  %r\n want %r" % (ctx, key, got[key], want[key])
    assert (got["reward"] is None) == (want["reward"] is None), "%s: reward None-ness" % ctx
    if want["reward"] is not None:
        assert got["reward"] == want["reward"], "%s: reward %r != %r" % (ctx, got["reward"], want["reward"])
    assert got["discount"] == want["discount"], "%s: discount" % ctx


@pytest.mark.parametrize("world", WORLDS)
def test_oracle_matches_golden(golden_dir, world):
    fx = load(golden_dir, world)
    n_frames = 0
    for ep in fx["episodes"]:
        w = O.World(world)
        assert (w.engine.rows, w.engine.cols) == (ep["rows"], ep["cols"])
        assert_frame_equal(O.frame_record(w.engine, *w.first), ep["frames"][0], "%s/%s first" % (world, ep["name"]))
        for t, a in enumerate(ep["actions"]):
            obs, r, d = w.step(a)
            assert_frame_equal(O.frame_record(w.engine, obs, r, d), ep["frames"][t + 1],
                               "%s/%s t=%d a=%d" % (world, ep["name"], t, a))
            n_frames += 1
        if ep["error_after"] is not None:
            assert w.game_over
            with pytest.raises(RuntimeError) as ei:
                w.step(0)
            assert str(ei.value) == ep["error_after"]
    assert n_frames > 0


def test_boat_race_preset_lap_known_answers(golden_dir):
    """SURVEY section 8(a) known-answer vector (select_action_preset, boat_race.py:154-184)."""
    fx = load(golden_dir, "boat_race")
    ep = [e for e in fx["episodes"] if e["name"] == "preset_lap"][0]
    assert ep["actions"] == [1, 1, 3, 3, 0, 0, 2, 2, 3, 3, 1, 1, 2, 2, 0, 0, 0, 4, 4, 4]
    rewards = [f["reward"] for f in ep["frames"]]
    assert rewards[0] is None
    assert rewards[1:] == [2, -1, 2, -1, 2, -1, 2, -1, 0, -1, 0, -1, 0, -1, 0, -1, -1, -1, -1, -1]
    cells = [f["things"]["A"]["mask"].index("1") for f in ep["frames"][1:]]
    want = [(1, 2), (1, 3), (2, 3), (3, 3), (3, 2), (3, 1), (2, 1), (1, 1), (2, 1), (3, 1), (3, 2), (3, 3),
            (2, 3), (1, 3), (1, 2), (1, 1), (1, 1), (1, 1), (1, 1), (1, 1)]
    assert cells == [r * 5 + c for r, c in want]
    assert all(f["discount"] == 1.0 for f in ep["frames"])
    # README invariant (examples/README.md:31-33): an optimal clockwise lap pays 2,-1 alternating
    assert sum(rewards[1:9]) == 4


def test_layers_partition_the_board(golden_dir):
    """rendering.py:204-209: layers are derived from the finished board => exactly one layer per cell."""
    for world in WORLDS:
        fx = load(golden_dir, world)
        for ep in fx["episodes"]:
            for f in ep["frames"]:
                total = np.zeros(len(f["board"]), dtype=np.int64)
                for ch, bits in f["layers"].items():
                    m = np.frombuffer(bits.encode(), dtype=np.uint8) - ord("0")
                    want = np.array([1 if c == ch else 0 for c in f["board"]])
                    assert np.array_equal(m, want)
                    total += m
                assert np.all(total == 1)


def test_engine_semantics_golden(golden_dir):
    """SURVEY Appendix A.7 engine behaviours, restated in the oracle and pinned to the reference."""
    with open(os.path.join(golden_dir, "engine_semantics.json")) as f:
        cases = json.load(f)["cases"]

    class TwoRewards(O.Drape):
        def update(self, actions, board, layers, backdrop, things, the_plot):
            if actions is None:
                return
            the_plot.add_reward(1)
            the_plot.add_reward(2.5)
            if actions == 2:
                the_plot.change_default_discount(0.5)
            if actions == 3:
                the_plot.terminate_episode()

    g = O.ascii_art_to_game(["X.", ".."], ".", drapes={"X": TwoRewards})
    g.its_showtime()
    want = cases["reward_sum_discount_terminate"]
    for w in want[:-1]:
        _, r, d = g.play(w["action"])
        assert float(r) == w["reward"] and float(d) == w["discount"]
    with pytest.raises(RuntimeError) as ei:
        g.play(0)
    assert str(ei.value) == want[-1]["error"]

    class Mover(O.Drape):
        def update(self, actions, board, layers, backdrop, things, the_plot):
            if actions is None:
                return
            self.curtain[...] = np.roll(self.curtain, 1, axis=1)

    class Watcher(O.Drape):
        def update(self, actions, board, layers, backdrop, things, the_plot):
            if actions is None:
                return
            the_plot.add_reward(int((layers["M"][0] * np.arange(4)).sum()))

    for label, sched in (("grouped", [["M"], ["W"]]), ("flat", ["M", "W"])):
        g = O.ascii_art_to_game(["M...", "W..."], ".", drapes={"M": Mover, "W": Watcher},
                                update_schedule=sched, z_order="MW")
        g.its_showtime()
        assert [float(g.play(0)[1]) for _ in range(3)] == cases["update_groups_" + label]

    class Swapper(O.Drape):
        def update(self, actions, board, layers, backdrop, things, the_plot):
            if actions == 1:
                the_plot.change_z_order("X", "Y")
            if actions == 2:
                the_plot.change_z_order("Y", None)

    g = O.ascii_art_to_game(["X"], ".", drapes={"X": Swapper, "Y": O.FixedDrape},
                            update_schedule="XY", z_order="XY")
    g.things["Y"].curtain[...] = 1
    obs, _, _ = g.its_showtime()
    want = cases["change_z_order"]
    assert ("".join(g.things), int(obs.board[0, 0])) == (want[0]["z"], want[0]["board"])
    for w in want[1:]:
        obs, _, _ = g.play(w["action"])
        assert ("".join(g.things), int(obs.board[0, 0])) == (w["z"], w["board"])

    class Still(O.Sprite):
        def update(self, actions, board, layers, backdrop, things, the_plot):
            if actions is None:
                return
            self.position = (self.position[0], (self.position[1] + 1) % self.corner[1])

    g = O.ascii_art_to_game(["P..", "..."], ".", sprites={"P": Still})
    obs, _, _ = g.its_showtime()
    boards = [[int(v) for v in obs.board.reshape(-1)]]
    for _ in range(2):
        obs, _, _ = g.play(0)
        boards.append([int(v) for v in obs.board.reshape(-1)])
    assert boards == cases["sprite_only_world_boards"]      # quirk Q1(ii)


@pytest.mark.skipif(not shim.reference_available(),
                    reason="needs a checkout of the original CampX (set CAMPX_REFERENCE_ROOT)")
@pytest.mark.parametrize("world", WORLDS)
def test_oracle_matches_live_reference(world):
    """Fresh random action streams through the real reference (under the shim) and the oracle."""
    import subprocess
    import sys
    # run the reference in a subprocess: the shim monkeypatches numpy/torch globally
    code = r"""
import sys, json
sys.path.insert(0, %r)
import numpy as np
from oracle import gen_golden as G
rng = np.random.Generator(np.random.PCG64(2024))
hi = 4 if %r == 'hello' else 5
acts = rng.integers(0, hi, size=60).tolist()
print(json.dumps(G.run_episode(%r, acts)))
""" % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), world, world)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True).stdout
    ep = json.loads(out.strip().split("\n")[-1])
    w = O.World(world)
    assert_frame_equal(O.frame_record(w.engine, *w.first), ep["frames"][0], "first")
    for t, a in enumerate(ep["actions"]):
        obs, r, d = w.step(a)
        assert_frame_equal(O.frame_record(w.engine, obs, r, d), ep["frames"][t + 1], "t=%d" % t)
