"""The compiler's fit of sprites that walls stop (PyColab's MazeWalker: CX_KIND_SPRITE with blockers), its refusals,
and every world that compiled before them unchanged.  Host only: no GPU."""
import pytest

from campx_b200 import _native as N
from campx_b200 import things
from campx_b200.ascii_art import Partial, ascii_art_to_game
from campx_b200.compiler import CompileError
from examples import generality_worlds, worlds
from examples.worlds import Coin, Runner
from tests.test_pickup_compile import PARENT_DIGESTS, _digest

MOVES = [(0, -1), (0, 1), (-1, 0), (1, 0), (0, 0)]


def _agent(spec):
    return {e.character: e for e in spec.entities}['A']


@pytest.mark.parametrize("name", ["maze", "sprite_race"])
def test_runner_fits_moves_and_blockers(name):
    spec = worlds.make_world(name).compile()
    a = _agent(spec)
    assert a.kind == N.CX_KIND_SPRITE and a.moves == MOVES and a.blockers == '#'
    assert a.visible_op == [N.CX_VIS_KEEP] * 5 and a.init_pos == (1, 1)
    summary = _agent(spec).summary()
    assert summary["kind"] == "sprite" and summary["blockers"] == '#' and summary["moves"] == MOVES
    assert {e["char"]: e for e in spec.summary()["entities"]}['A'] == summary
    d, _ = spec.to_ctypes()
    z = [e.character for e in spec.entities].index('A')
    assert d.entities[z].kind == N.CX_KIND_SPRITE and d.entities[z].blockers == 1 << spec.chars.index('#')


def test_maze_rewards_and_exit_watch_the_sprite():
    spec = worlds.make_world('maze').compile()
    ents = {e.character: e for e in spec.entities}
    assert ents['A'].step_reward == [-0.25] * 5
    assert ents['*'].watch == 'A' and all(v == {'*': 1.0} for v in ents['*'].entry_reward.values())
    assert ents['E'].watch == 'A' and all(v == {'E': 0.0} for v in ents['E'].terminate_on.values())


def test_a_blocker_in_the_backdrop():
    """'~' is scenery, not a drape: the sprite still stops at it (and, first in z-order, stamps the backdrop)."""
    art = ['######', '#A ~ #', '# #  #', '#~   #', '######']
    spec = ascii_art_to_game(art, ' ', sprites={'A': Partial(Runner, walls='#~')}, drapes={'#': things.FixedDrape},
                             z_order='A#').compile()
    assert _agent(spec).blockers == '#~' and _agent(spec).moves == MOVES


class Fader(Runner):
    """A Runner that hides itself whenever a wall stops it."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        before = self.position
        super(Fader, self).update(actions, board, layers, backdrop, all_things, the_plot)
        if actions is not None and int(actions.argmax()) != 4 and self.position == before:
            self._visible = False


class Skater(things.Sprite):
    """Moves right by one cell on the left half of the board and by two on the right half."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        step = 1 if self.position.col < self.corner.col // 2 else 2
        self._position = self.Position(self.position.row, (self.position.col + step) % self.corner.col)


class Ducker(Runner):
    """A Runner that hides every time it moves right: a blocked sprite may not change its visibility."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        super(Ducker, self).update(actions, board, layers, backdrop, all_things, the_plot)
        if actions is not None and int(actions.argmax()) == 1:
            self._visible = not self._visible


ROOM = ['#######', '#A    #', '#  #  #', '#######']


def test_refuses_a_blocked_sprite_that_changes_its_visibility():
    g = ascii_art_to_game(ROOM, ' ', sprites={'A': Partial(Ducker, walls='#')}, drapes={'#': things.FixedDrape},
                          z_order='#A')
    with pytest.raises(CompileError, match=r"sprite 'A' does not move by a fixed toroidal displacement .* a sprite "
                                           r"that walls stop must keep its visibility"):
        g.compile()
    g = ascii_art_to_game(ROOM, ' ', sprites={'A': Partial(Fader, walls='#')}, drapes={'#': things.FixedDrape},
                          z_order='#A')
    with pytest.raises(CompileError, match=r"sprite 'A'"):
        g.compile()


def test_refuses_moves_that_differ_by_position():
    g = ascii_art_to_game(['S.......', '........'], '.', sprites={'S': Skater}, action_format="index")
    with pytest.raises(CompileError, match=r"sprite 'S': action \d moves it by different amounts"):
        g.compile()


def test_refuses_pickups_with_a_sprite_agent():
    g = ascii_art_to_game(worlds.COINS_ART, ' ', sprites={'A': Partial(Runner, walls='#')},
                          drapes={'$': Coin, '#': things.FixedDrape}, z_order='$A#', update_schedule='A$#')
    with pytest.raises(CompileError, match=r"pickup drape '\$' needs a single-agent game"):
        g.compile()


@pytest.mark.parametrize("name", sorted(PARENT_DIGESTS))
def test_worlds_compile_to_the_same_bytes(name):
    if name in ('boat_race', 'demo1', 'demo2', 'demo3', 'demo4', 'hello'):
        spec = worlds.make_world(name).compile()
    else:
        spec = generality_worlds.make_generality_world(name).compile()
    assert _digest(spec) == PARENT_DIGESTS[name]
