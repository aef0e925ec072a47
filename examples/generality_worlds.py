"""Three small worlds that use the engine features none of CampX's own worlds touch (SURVEY 8(f) row 3):

    zswap    `the_plot.change_z_order(...)` directives          campx/plot.py:121-159, engine.py:242-281,163
    ghost    sprites that hide and show themselves              campx/things.py:320,390-392, engine.py:315
    scroll   a `Backdrop` subclass whose `update()` scrolls it  campx/things.py:103-148

plus two "reach the goal" worlds (ADVICE r1: `terminate_episode` that depends on where the agent stands):

    goal     an agent, an exit `G` (reward 10, episode over) and a pit `X` (reward -5, over with discount 0.25)
    goal2    the same with a drifting sprite, so that the game runs on the generic kernels

written, like examples/worlds.py, as ordinary single-environment `Sprite` / `Drape` / `Backdrop`
subclasses.  The same three worlds exist against the reference API (oracle/gen_golden.py, executed on the
unmodified reference to record tests/golden/generality_*.json) and as numpy oracle entities
(oracle/campx_oracle.py); the GPU tests compare all of them frame by frame.  They also cover the interplay
with quirk Q1: which sprites stamp their character into the backdrop depends on the CURRENT z-order and
visibility.
"""
import numpy as np
import torch

from campx_b200 import things
from campx_b200.ascii_art import ascii_art_to_game, Partial
from examples.worlds import Walker, cells_of

ZSWAP_ART = ['S.....',
             '.XX.Y.',
             '.XXYY.',
             '...YY.',
             '......']

GHOST_ART = ['G..@.',
             '..@..',
             'H....']

SCROLL_ART = ['A.~~.^',
              '.~..^.',
              '~..^..',
              '..^..~']


GOAL_ART = ['######',
            '#A  G#',
            '# #  #',
            '#   X#',
            '######']

GOAL2_ART = ['######',
             '#A  G#',
             '# #  #',
             '#S  X#',
             '######']


def _rolled(curtain, shift, axis):
    return torch.from_numpy(np.roll(curtain.numpy(), shift, axis).copy())


class Shuffler(things.Drape):
    """Slides right on action 0; actions 1-3 reorder the z-order."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        if actions == 0:
            self.curtain.set_(_rolled(self.curtain, 1, 1))
            the_plot.add_reward(1)
        elif actions == 1:
            the_plot.change_z_order('X', 'Y')
        elif actions == 2:
            the_plot.change_z_order('Y', None)
        elif actions == 3:
            the_plot.change_z_order('X', None)
            the_plot.change_z_order('Y', 'X')


class Climber(things.Sprite):
    """Moves right / down; action 4 brings it to the front, action 2 sends it to the back."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        row, col = self.position
        if actions == 0:
            col = (col + 1) % self.corner.col
        elif actions == 1:
            row = (row + 1) % self.corner.row
        self._position = self.Position(row, col)
        if actions == 4:
            the_plot.change_z_order('S', 'Y')
        elif actions == 2:
            the_plot.change_z_order('S', None)


class Phantom(things.Sprite):
    """A sprite that can hide: action 4 toggles; `switchable` ones also hide on 2 and show on 3."""

    def __init__(self, corner, position, character, start_visible, d_row, d_col, switchable):
        super(Phantom, self).__init__(corner, position, character)
        self._visible = start_visible
        self._step = (d_row, d_col)
        self._switchable = switchable

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        row, col = self.position
        if actions == 0:
            col = (col + self._step[1]) % self.corner.col
        elif actions == 1:
            row = (row + self._step[0]) % self.corner.row
        self._position = self.Position(row, col)
        if self._switchable and actions in (2, 3):
            self._visible = actions == 3
        if actions == 4:
            self._visible = not self._visible


class Drizzle(things.Drape):
    """Falls one row on action 1; pays 0.5 every step."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        if actions == 1:
            self.curtain.set_(_rolled(self.curtain, 1, 0))
        the_plot.add_reward(0.5)


class Panorama(things.Backdrop):
    """Scenery that scrolls one cell in the direction of the (one-hot) action."""
    SCROLL = ((-1, 1), (1, 1), (-1, 0), (1, 0))      # (shift, axis) for left, right, up, down

    def update(self, actions, board, layers, all_things, the_plot):
        if actions is None:
            return
        a = int(torch.as_tensor(actions).argmax())
        if a < 4:
            shift, axis = self.SCROLL[a]
            self.curtain.set_(_rolled(self.curtain, shift, axis))


class Exit(things.Drape):
    """A cell that ends the episode when the agent steps onto it: pays `prize` and calls
    `terminate_episode(pcontinue)` (plot.py:161-184) -- the PyColab "reach the goal" idiom, written the way
    boat_race's tiles watch the agent (boat_race.py:79-82)."""

    def __init__(self, curtain, character, prize, pcontinue=0.0, agent='A'):
        super(Exit, self).__init__(curtain, character)
        self.prize, self.pcontinue, self.agent = prize, pcontinue, agent

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        here = (cells_of(all_things[self.agent], self.curtain) * layers[self.character]).sum()
        the_plot.add_reward(here * self.prize)
        if here > 0:
            the_plot.terminate_episode(self.pcontinue)


class Drifter(things.Sprite):
    """Moves one cell to the right (toroidally) every step."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        self._position = self.Position(self.position.row, (self.position.col + 1) % self.corner.col)


def make_generality_world(name, **engine_kwargs):
    """Un-started Engine for one of: zswap, ghost, scroll, goal, goal2."""
    if name in ('goal', 'goal2'):
        drapes = {'A': Partial(Walker, walls='#', per_step=-1, strict=True), '#': things.FixedDrape,
                  'G': Partial(Exit, 10), 'X': Partial(Exit, -5, 0.25)}
        if name == 'goal':
            return ascii_art_to_game(GOAL_ART, ' ', drapes=drapes, update_schedule='AGX#', z_order='GXA#',
                                     **engine_kwargs)
        return ascii_art_to_game(GOAL2_ART, ' ', sprites={'S': Drifter}, drapes=drapes,
                                 update_schedule='ASGX#', z_order='GXAS#', **engine_kwargs)
    if name == 'zswap':
        return ascii_art_to_game(ZSWAP_ART, '.', sprites={'S': Climber},
                                 drapes={'X': Shuffler, 'Y': things.FixedDrape},
                                 update_schedule='SXY', z_order='SXY', **engine_kwargs)
    if name == 'ghost':
        return ascii_art_to_game(GHOST_ART, '.',
                                 sprites={'G': Partial(Phantom, True, 1, 1, True),
                                          'H': Partial(Phantom, False, 1, -1, False)},
                                 drapes={'@': Drizzle}, update_schedule='GH@', z_order='GH@', **engine_kwargs)
    if name == 'scroll':
        return ascii_art_to_game(SCROLL_ART, '.',
                                 drapes={'A': Partial(Walker, walls='^', per_step=1, strict=True)},
                                 backdrop=Panorama, z_order='A', **engine_kwargs)
    raise KeyError(name)
