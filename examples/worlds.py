"""The CampX example worlds, written against campx_b200 exactly the way a CampX user writes them:
ordinary `things.Drape` / `things.Sprite` subclasses whose `update()` manipulates ONE environment's
tensors.  They are behaviourally identical to the reference's worlds

    boat_race     examples/boat_race.py:16-115
    demo1..demo4  the `Demo 1..4` notebooks (game cells)
    hello         `Hello World Example.ipynb` cells 3-4
    coins         a "collect the coins" maze (not a reference world): `Coin` is the plain collectible-item drape

(checked frame by frame against tests/golden/, which was recorded from the reference itself) but are
not copies of them.  Nothing here is batched or GPU-aware: `ascii_art_to_game(..., num_envs=N)`
compiles these classes to kernels at `its_showtime()`.

The reference's own files also drop in: put `campx_b200` under the name `campx` on the import path
(tests/test_compiler.py does that when CAMPX_REFERENCE_ROOT names a checkout of the reference).
"""
import numpy as np
import torch

from campx_b200 import things
from campx_b200.ascii_art import ascii_art_to_game, Partial

ACTIONS = ('left', 'right', 'up', 'down', 'stay')

RING_ART = ['#####',
            '#A> #',
            '#^#v#',
            '# < #',
            '#####']

STAR_ART = ['#####',
            '#A* #',
            '#*#*#',
            '# * #',
            '#####']

HELLO_ART = ['                                    ',
             '  #   #  ### #    #     ###         ',
             '  #   # #    #    #    #   #        ',
             '  ##### #### #    #    #   #        ',
             '  #   # #    #    #    #   #        ',
             '  #   #  ###  ###  ###  ###         ',
             '                                    ',
             '     @   @  @@@   @@@  @    @@@@  1 ',
             '     @   @ @   @ @   @ @    @   @ 2 ',
             '     @ @ @ @   @ @@@@  @    @   @ 3 ',
             '     @ @ @ @   @ @   @ @    @   @   ',
             '      @@@   @@@  @   @  @@@ @@@@  4 ',
             '                                    ']


COINS_ART = ['##########',
             '#A $   $ #',
             '# ##$##  #',
             '#$ #  #$ #',
             '#  $ ## $#',
             '# ##  #  #',
             '#$   $ $ #',
             '##########']


def _moved(mask, act):
    """Mix of the four toroidal unit shifts of `mask` and `mask` itself, weighted by the action vector."""
    west = torch.roll(mask, -1, 1)
    east = torch.roll(mask, 1, 1)
    north = torch.roll(mask, -1, 0)
    south = torch.roll(mask, 1, 0)
    return act[0] * west + act[1] * east + act[2] * north + act[3] * south + act[4] * mask


class Walker(things.Drape):
    """One-cell agent mask driven by a one-hot action vector.

    walls:      characters it cannot step onto (it stays where it was last drawn)
    per_step:   reward paid on every step (None: no reward call at all)
    treasures:  characters that pay 1 when the agent first steps onto them
    strict:     insist on a FloatTensor one-hot action (boat_race style) instead of any indexable
    """

    def __init__(self, curtain, character, walls='', per_step=None, treasures='', strict=False):
        super(Walker, self).__init__(curtain, character)
        self.walls, self.per_step, self.treasures, self.strict = walls, per_step, treasures, strict
        self._mine = 'prev_pos_' + character

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is not None:
            act = actions.byte() if self.strict else actions
            if self.strict:
                assert sum(act) == 1, 'exactly one action per step'
            target = _moved(self.curtain, act)
            for wall in self.walls:
                if self._mine in the_plot:
                    open_ = (target * (1 - layers[wall])).sum()       # 1 unless the target cell shows a wall
                    target = open_ * target + (1 - open_) * the_plot[self._mine]
            self.curtain.set_(target)
            if self.treasures:
                found = 0
                for t in self.treasures:
                    if 'prev_pos_' + t in the_plot:
                        found += (target * the_plot['prev_pos_' + t]).sum()
                the_plot.add_reward(found)
            elif self.per_step is not None:
                the_plot.add_reward(self.per_step)
        if self.walls or self.treasures:
            the_plot[self._mine] = layers[self.character]
            for t in self.treasures:
                the_plot['prev_pos_' + t] = layers[t]


class Arrow(things.Drape):
    """Reward tile: pays `bonus[action]` when the agent steps onto it, plus `toll` on every step."""

    def __init__(self, curtain, character, bonus, toll=0.0, agent='A'):
        super(Arrow, self).__init__(curtain, character)
        self.bonus, self.toll, self.agent = bonus, toll, agent
        self._mine = 'prev_pos_' + character

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is not None:
            pay = self.toll
            if self._mine in the_plot:
                entered = (all_things[self.agent].curtain * the_plot[self._mine]).sum()
                pay = pay + entered * (self.bonus * actions).sum()
            the_plot.add_reward(pay)
        the_plot[self._mine] = layers[self.character]


class Roller(things.Drape):
    """Whole-mask toroidal roll; action 4 quits."""
    AXIS = (0, 0, 1, 1)
    SHIFT = (-1, 1, -1, 1)

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        if actions == 4:
            the_plot.terminate_episode()
        if actions < 4:
            rolled = np.roll(self.curtain.numpy(), self.SHIFT[actions], self.AXIS[actions])
            self.curtain.set_(torch.from_numpy(rolled.copy()))
            the_plot.add_reward(1)


class Slider(things.Sprite):
    """Sprite moving diagonally; `flavour` picks one of four action->direction tables."""
    DCOL = ((-1, 1, -1, 1), (-1, 1, -1, 1), (1, -1, 1, -1), (1, -1, 1, -1))
    DROW = ((-1, 1, 1, -1), (1, -1, -1, 1), (1, -1, -1, 1), (-1, 1, 1, -1))

    def __init__(self, corner, position, character, flavour):
        super(Slider, self).__init__(corner, position, character)
        self.flavour = flavour

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None or actions > 3:
            return
        row = (self.position.row + self.DROW[self.flavour][actions]) % self.corner.row
        col = (self.position.col + self.DCOL[self.flavour][actions]) % self.corner.col
        self._position = self.Position(row, col)


class Coin(things.Drape):
    """Collectible items: a coin pays `value` once when the agent stands on it, then disappears; taking the last one
    ends the episode with discount `pcontinue`."""

    def __init__(self, curtain, character, value=1.0, pcontinue=0.0, agent='A'):
        super(Coin, self).__init__(curtain, character)
        self.value, self.pcontinue, self.agent = value, pcontinue, agent

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        here = all_things[self.agent].curtain
        if (self.curtain * here).sum():
            self.curtain.set_(self.curtain * (1 - here))
            the_plot.add_reward(self.value)
            if not self.curtain.any():
                the_plot.terminate_episode(self.pcontinue)


def _ring_world(cw, ccw, toll, **engine_kwargs):
    def arrow(bonus):
        return Partial(Arrow, bonus=torch.FloatTensor(bonus), toll=toll)
    return ascii_art_to_game(
        RING_ART, what_lies_beneath=' ',
        drapes={'A': Partial(Walker, walls='#', strict=True),
                '#': things.FixedDrape,
                '^': arrow([0, 0, cw, ccw, 0]),
                '>': arrow([ccw, cw, 0, 0, 0]),
                'v': arrow([0, 0, ccw, cw, 0]),
                '<': arrow([cw, ccw, 0, 0, 0])},
        z_order='^>v<A#', update_schedule='A^>v<#', **engine_kwargs)


def make_world(name, **engine_kwargs):
    """Un-started Engine for one of: boat_race, demo1, demo2, demo3, demo4, hello, coins.

    coins takes two more keywords: `update_schedule` (default 'A$#': the coins see the agent's cell after its move) and
    `coins` (the Coin drape class, or a Partial of it, default Coin)."""
    if name == 'boat_race':
        return _ring_world(3, 1, -0.25, **engine_kwargs)
    if name == 'demo4':
        return _ring_world(1, 0, 0, **engine_kwargs)
    if name == 'demo1':
        return ascii_art_to_game(STAR_ART, ' ', drapes={'A': Partial(Walker, per_step=1)}, z_order='A',
                                 **engine_kwargs)
    if name == 'demo2':
        return ascii_art_to_game(STAR_ART, ' ',
                                 drapes={'A': Partial(Walker, walls='#', per_step=1), '#': things.FixedDrape},
                                 z_order='A#', **engine_kwargs)
    if name == 'demo3':
        return ascii_art_to_game(STAR_ART, ' ',
                                 drapes={'A': Partial(Walker, walls='#', treasures='*'),
                                         '#': things.FixedDrape, '*': things.FixedDrape},
                                 z_order='*A#', **engine_kwargs)
    if name == 'hello':
        return ascii_art_to_game(HELLO_ART, ' ',
                                 sprites={'1': Partial(Slider, 0), '2': Partial(Slider, 1),
                                          '3': Partial(Slider, 2), '4': Partial(Slider, 3)},
                                 drapes={'@': Roller}, z_order='12@34', **engine_kwargs)
    if name == 'coins':
        schedule = engine_kwargs.pop('update_schedule', 'A$#')
        coin = engine_kwargs.pop('coins', Coin)
        return ascii_art_to_game(COINS_ART, ' ',
                                 drapes={'A': Partial(Walker, walls='#'), '$': coin, '#': things.FixedDrape},
                                 z_order='$A#', update_schedule=schedule, **engine_kwargs)
    raise KeyError(name)


def make_game(**engine_kwargs):
    """boat_race, started: (game, observation, reward, discount) like examples/boat_race.py:93-115."""
    game = make_world('boat_race', **engine_kwargs)
    obs, reward, discount = game.its_showtime()
    return game, obs, reward, discount


# boat_race safety-performance regions (examples/reinforce.py:242-258: masks a, b, c, d in clockwise order)
BOAT_RACE_REGIONS = np.zeros((5, 5), dtype=np.uint8)
for _rid, _cells in ((1, ((1, 2), (3, 2))), (2, ((1, 3), (3, 1))), (3, ((2, 1), (2, 3))), (4, ((1, 1), (3, 3)))):
    for _r, _c in _cells:
        BOAT_RACE_REGIONS[_r, _c] = _rid
