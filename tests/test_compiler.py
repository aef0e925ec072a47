"""Game compiler (host side, no GPU): fingerprinting user entity classes into kernel primitives."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from campx_b200 import things
from campx_b200.ascii_art import ascii_art_to_game, Partial
from campx_b200.compiler import CompileError
from examples.worlds import make_world
from oracle import shim
from tests.expected_specs import expected_spec

WORLDS = ["boat_race", "demo1", "demo2", "demo3", "demo4", "hello"]


def assert_same_spec(got, want):
    assert got.summary() == want.summary()
    assert np.array_equal(np.asarray(got.backdrop), np.asarray(want.backdrop))
    for a, b in zip(got.entities, want.entities):
        assert np.array_equal(np.asarray(a.mask) != 0, np.asarray(b.mask) != 0), a.character


@pytest.mark.parametrize("world", WORLDS)
def test_example_worlds_compile_to_expected_primitives(world):
    spec = make_world(world, num_envs=8).compile()
    assert_same_spec(spec, expected_spec(world))
    spec.to_ctypes()


def test_compile_is_idempotent_and_freezes_setup():
    g = make_world("boat_race", num_envs=2)
    assert g.compile() is g.compile()
    with pytest.raises(RuntimeError):
        g.update_group("x")                      # engine.py:327-330: no set-up after showtime


def test_action_format_detection():
    assert make_world("boat_race").compile().action_format == "onehot_float"
    assert make_world("hello").compile().action_format == "index"
    with pytest.raises(CompileError):
        make_world("hello", action_format="onehot_float").compile()


def test_unsupported_behaviour_is_refused_not_approximated():
    class Grower(things.Drape):                  # mask grows: neither static, one-cell move nor roll
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is not None:
                self.curtain[0, 0] = 1

    g = ascii_art_to_game(["..G", "..G"], ".", drapes={"G": Grower}, action_format="index")
    with pytest.raises(NotImplementedError):
        g.compile()

    class Zed(things.Drape):                     # engine.py:270-279 would drop 'Z' from the game altogether
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions == 1:
                the_plot.change_z_order("Z", "Z")

    g = ascii_art_to_game(["Z."], ".", drapes={"Z": Zed}, action_format="index")
    with pytest.raises((NotImplementedError, KeyError)):
        g.compile()

    class Blinker(things.Sprite):                # visibility depends on the position, not only on the action
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is not None:
                self._position = self.Position(self.position.row, (self.position.col + 1) % self.corner.col)
                self._visible = self.position.row == 0

    g = ascii_art_to_game(["B...", "...."], ".", sprites={"B": Blinker}, action_format="index")
    with pytest.raises(NotImplementedError):
        g.compile()

    class Painter(things.Backdrop):              # the backdrop changes, but not by a roll
        def update(self, actions, board, layers, all_things, the_plot):
            if actions is not None:
                self.curtain[0, 0] = ord("x")

    g = ascii_art_to_game(["W.x", "..."], ".", drapes={"W": things.FixedDrape}, backdrop=Painter,
                          action_format="index")
    with pytest.raises(NotImplementedError):
        g.compile()

    class StateDependentReward(things.Drape):    # reward depends on the frame counter
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is not None:
                the_plot.add_reward(the_plot.frame % 2)

    g = ascii_art_to_game(["S."], ".", drapes={"S": StateDependentReward}, action_format="index")
    spec = g.compile()       # constant over the probes (all taken at the same frame): accepted here ...
    assert spec.entities[0].step_reward is not None
    # ... and caught by the on-device replay in its_showtime (tests/test_gpu_engine.py)


def test_custom_world_with_two_groups_and_discount():
    class Hopper(things.Sprite):
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is None:
                return
            if actions == 2:
                the_plot.change_default_discount(0.5)
            if actions == 3:
                the_plot.terminate_episode(0.25)
            step = (0, 1) if actions == 0 else (0, -1) if actions == 1 else (0, 0)
            self._position = self.Position((self.position.row + step[0]) % self.corner.row,
                                           (self.position.col + step[1]) % self.corner.col)
            the_plot.add_reward(2.5)

    g = ascii_art_to_game(["H..", "###"], ".", sprites={"H": Hopper}, drapes={"#": things.FixedDrape},
                          update_schedule=[["H"], ["#"]], z_order="#H", num_actions=4)
    spec = g.compile()
    s = spec.summary()
    assert s["n_groups"] == 2 and s["action_format"] == "index"
    h = [e for e in s["entities"] if e["char"] == "H"][0]
    assert h["moves"] == [(0, 1), (0, -1), (0, 0), (0, 0)]
    assert h["step_reward"] == [2.5] * 4
    assert h["terminate"] == {3: 0.25} and h["discount"] == {2: 0.5}


def test_engine_generality_primitives():
    """SURVEY 8(f) row 3: z-order directives, sprite visibility and a scrolling backdrop are fitted per action."""
    from examples.generality_worlds import make_generality_world
    s = make_generality_world("zswap").compile().summary()
    x = [e for e in s["entities"] if e["char"] == "X"][0]
    assert x["z_orders"] == {1: [("X", "Y")], 2: [("Y", None)], 3: [("X", None), ("Y", "X")]}
    s = make_generality_world("ghost").compile().summary()
    g = [e for e in s["entities"] if e["char"] == "G"][0]
    assert g["visible_op"] == ["keep", "keep", "hide", "show", "toggle"] and g["visible"] is True
    h = [e for e in s["entities"] if e["char"] == "H"][0]
    assert h["visible"] is False and h["visible_op"][4] == "toggle"
    s = make_generality_world("scroll").compile().summary()
    assert s["backdrop_moves"] == [(0, -1), (0, 1), (-1, 0), (1, 0), (0, 0)]


def test_reach_the_goal_games_compile_to_conditional_terminate():
    """ADVICE r1: terminate_episode that depends on where the agent stands is fitted per (action, character under the
    watched entity), like entry rewards; the pit passes its own discount."""
    from examples.generality_worlds import make_generality_world
    for world in ("goal", "goal2"):
        s = make_generality_world(world).compile().summary()
        ent = {e["char"]: e for e in s["entities"]}
        assert ent["G"]["watch"] == "A" and ent["G"]["terminate_on"] == {1: {"G": 0.0}, 2: {"G": 0.0}}
        assert ent["G"]["entry_reward"] == {1: {"G": 10.0}, 2: {"G": 10.0}} and "terminate" not in ent["G"]
        assert ent["X"]["terminate_on"] == {1: {"X": 0.25}, 3: {"X": 0.25}}
        assert ent["A"]["blockers"] == "#" and ent["A"]["step_reward"] == [-1.0] * 5
    # the C ABI receives them as per-action character bit sets
    desc, keep = make_generality_world("goal").compile().to_ctypes()
    chars = make_generality_world("goal").compile().chars
    g = [desc.entities[z] for z in range(desc.n_entities) if chr(desc.entities[z].character) == "G"][0]
    assert [g.terminate_chars[a] for a in range(5)] == [0, 1 << chars.index("G"), 1 << chars.index("G"), 0, 0]
    assert g.terminate_value[1] == 0.0


def test_hidden_state_is_refused():
    """ADVICE r1: probes start from a copy of the first frame, so an entity that counts its own steps would look
    stateless and compile to a game that pays the wrong rewards later.  Instance attributes and non-tensor Plot
    entries that change during a step are detected and the game is refused."""
    from campx_b200.compiler import CompileError

    class Metronome(things.Drape):
        def __init__(self, curtain, character):
            super(Metronome, self).__init__(curtain, character)
            self.n = 0

        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is None:
                return
            self.n += 1
            the_plot.add_reward(5 if self.n % 40 == 0 else 0)

    g = ascii_art_to_game(["M.", ".."], ".", drapes={"M": Metronome})
    with pytest.raises(CompileError) as ei:
        g.compile()
    assert "'n'" in str(ei.value) and "'M'" in str(ei.value)

    class PlotCounter(things.Drape):
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is None:
                return
            the_plot["ticks"] = the_plot.get("ticks", 0) + 1
            the_plot.add_reward(1 if the_plot["ticks"] > 30 else 0)

    g = ascii_art_to_game(["M.", ".."], ".", drapes={"M": PlotCounter})
    with pytest.raises(CompileError) as ei:
        g.compile()
    assert "ticks" in str(ei.value)

    class Harmless(things.Drape):                 # attributes that never change are not state
        def __init__(self, curtain, character):
            super(Harmless, self).__init__(curtain, character)
            self.bonus, self.table = 2, [1, 2, 3]

        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is not None:
                the_plot.add_reward(self.bonus)

    assert ascii_art_to_game(["M.", ".."], ".", drapes={"M": Harmless}).compile().entities[0].step_reward == [2.0] * 5


REFERENCE_EXAMPLES = os.path.join(shim.REFERENCE_ROOT, "examples")
NEEDS_REFERENCE = pytest.mark.skipif(not shim.reference_available("examples"),
                                     reason="needs a checkout of the original CampX (set CAMPX_REFERENCE_ROOT)")


@NEEDS_REFERENCE
def test_reference_boat_race_file_drops_in_unchanged(monkeypatch):
    """The reference's own examples/boat_race.py, imported with campx_b200 standing in for campx,
    compiles to exactly the primitives of our boat_race world (hence runs identically on the GPU)."""
    import campx_b200
    import campx_b200.ascii_art
    import campx_b200.engine
    alias = types.ModuleType("campx")
    alias.things = campx_b200.things
    alias.ascii_art = campx_b200.ascii_art
    alias.engine = campx_b200.engine
    for name, mod in (("campx", alias), ("campx.things", campx_b200.things),
                      ("campx.ascii_art", campx_b200.ascii_art), ("campx.engine", campx_b200.engine)):
        monkeypatch.setitem(sys.modules, name, mod)
    monkeypatch.syspath_prepend(REFERENCE_EXAMPLES)
    monkeypatch.delitem(sys.modules, "boat_race", raising=False)
    captured = []

    def fake_showtime(self):                      # no GPU here: stop after the compile step
        captured.append(self)
        self.compile()
        return None, None, 1.0

    monkeypatch.setattr(campx_b200.engine.Engine, "its_showtime", fake_showtime)
    import boat_race as ref_boat_race
    assert ref_boat_race.__file__.startswith(REFERENCE_EXAMPLES)
    game, _, _, _ = ref_boat_race.make_game()
    assert_same_spec(game.spec, expected_spec("boat_race"))


@NEEDS_REFERENCE
@pytest.mark.parametrize("world,notebook", [
    ("demo1", "Demo 1: Simple Agent Example.ipynb"),
    ("demo2", "Demo 2: Simple Wall Example.ipynb"),
    ("demo3", "Demo 3: Hover Reward Example.ipynb"),
    ("demo4", "Demo 4: Directional Hover Reward Example.ipynb"),
    ("demo4", "Demo 5: Boat Race Example.ipynb"),       # the notebook's world carries Demo 4's 0/1 rewards, no step penalty
    ("hello", "Hello World Example.ipynb"),
])
def test_reference_notebook_worlds_drop_in_unchanged(monkeypatch, world, notebook):
    """Game-defining cells of the reference notebooks, exec'd against campx_b200 under the name campx."""
    import json
    import campx_b200
    import campx_b200.ascii_art
    import campx_b200.engine
    alias = types.ModuleType("campx")
    alias.things, alias.ascii_art, alias.engine = campx_b200.things, campx_b200.ascii_art, campx_b200.engine
    for name, mod in (("campx", alias), ("campx.things", campx_b200.things),
                      ("campx.ascii_art", campx_b200.ascii_art), ("campx.engine", campx_b200.engine)):
        monkeypatch.setitem(sys.modules, name, mod)

    def fake_showtime(self):
        self.compile()
        return None, None, 1.0

    monkeypatch.setattr(campx_b200.engine.Engine, "its_showtime", fake_showtime)
    with open(os.path.join(REFERENCE_EXAMPLES, notebook)) as f:
        nb = json.load(f)
    ns = {"__name__": "nb"}
    for cell in nb["cells"]:
        src = "".join(cell["source"])
        if cell["cell_type"] != "code" or not any(t in src for t in ("class ", "def ", "import ", "_ART")):
            continue
        src = "\n".join(l for l in src.split("\n")
                        if not (not l.startswith(" ") and "= make_game()" in l) and "import curses" not in l
                        and not l.strip().startswith("import os, sys, curses")
                        # the PySyft worker preamble of Demo 3 (remote execution is out of scope, north_star)
                        and not any(t in l for t in ("syft", "hook", "VirtualWorker", "me.add_worker", "me.is_client_worker")))
        if "curses" in "".join(cell["source"]):
            src = "import os, sys, torch, six, itertools, collections\nimport numpy as np\n" + src
        exec(compile(src, notebook, "exec"), ns)
        if "make_game" in ns:
            break                                   # what follows is the notebook's RL / plotting code
    out = ns["make_game"]()
    game = out[0] if isinstance(out, tuple) else out
    spec = game.compile()
    want = expected_spec(world)
    if world in ("demo2", "hello"):
        # these notebooks leave update_schedule to the default; ours is sorted order (documented)
        assert {e.character: e.summary() | {"rank": 0} for e in spec.entities} == \
               {e.character: e.summary() | {"rank": 0} for e in want.entities}
    else:
        assert_same_spec(spec, want)
