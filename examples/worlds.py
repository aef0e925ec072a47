"""The CampX example worlds, written against campx_b200 exactly the way a CampX user writes them:
ordinary `things.Drape` / `things.Sprite` subclasses whose `update()` manipulates ONE environment's
tensors.  They are behaviourally identical to the reference's worlds

    boat_race     examples/boat_race.py:16-115
    demo1..demo4  the `Demo 1..4` notebooks (game cells)
    hello         `Hello World Example.ipynb` cells 3-4
    coins         a "collect the coins" maze (not a reference world): `Coin` is the plain collectible-item drape
    doorkey       MiniGrid's DoorKey (not a reference world): take the key `k` (a `Coin` worth nothing), the `Door`
                  opens, walk through to the exit; doorkey2 has two keys and two doors in a row
    maze          a sprite agent (`Runner`, PyColab's MazeWalker pattern) in a maze of walls, with treasure tiles
                  and an exit (not a reference world)
    sprite_race   boat_race with `Runner` as its agent (not a reference world)

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


DOORKEY_ART = ['#########',
               '#A  #   #',
               '#   D   #',
               '# k #  E#',
               '#########']

DOORKEY2_ART = ['############',
                '#A  #  K#  #',
                '#   D   d E#',
                '# k #   #  #',
                '############']


MAZE_ART = ['##########',
            '#A   #  *#',
            '# ## # # #',
            '#  #   # #',
            '## ### # #',
            '#*   #  E#',
            '##########']


def cells_of(thing, like):
    """The cells `thing` covers, as a mask shaped like `like`: a drape's curtain, or a sprite's one position."""
    if isinstance(thing, things.Sprite):
        mask = torch.zeros_like(like)
        mask[thing.position.row, thing.position.col] = 1
        return mask
    return thing.curtain


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
                entered = (cells_of(all_things[self.agent], self.curtain) * the_plot[self._mine]).sum()
                pay = pay + entered * (self.bonus * actions).sum()
            the_plot.add_reward(pay)
        the_plot[self._mine] = layers[self.character]


class Runner(things.Sprite):
    """A sprite agent that walks one cell per one-hot action (left, right, up, down, stay; toroidal) and does not step
    onto a cell that shows one of `walls` (PyColab's MazeWalker).

    per_step:   reward paid on every step (None: no reward call at all)
    """
    DROW = (0, 0, -1, 1, 0)
    DCOL = (-1, 1, 0, 0, 0)

    def __init__(self, corner, position, character, walls='', per_step=None):
        super(Runner, self).__init__(corner, position, character)
        self.walls, self.per_step = walls, per_step

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        a = int(np.argmax(np.asarray(actions, dtype=np.float32)))
        row = (self.position.row + self.DROW[a]) % self.corner.row
        col = (self.position.col + self.DCOL[a]) % self.corner.col
        if not any(int(layers[wall][row, col]) for wall in self.walls):
            self._position = self.Position(row, col)
        if self.per_step is not None:
            the_plot.add_reward(self.per_step)


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
    ends the episode with discount `pcontinue` (None: it does not end the episode, e.g. a key)."""

    def __init__(self, curtain, character, value=1.0, pcontinue=0.0, agent='A'):
        super(Coin, self).__init__(curtain, character)
        self.value, self.pcontinue, self.agent = value, pcontinue, agent

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        here = cells_of(all_things[self.agent], self.curtain)
        if (self.curtain * here).sum():
            self.curtain.set_(self.curtain * (1 - here))
            the_plot.add_reward(self.value)
            if not self.curtain.any() and self.pcontinue is not None:
                the_plot.terminate_episode(self.pcontinue)


class Door(things.Drape):
    """A door locked by the key drape `key`: it opens (its whole curtain clears) in the first step that finds every key
    taken, and stays open for the rest of the episode.  It must update after its key."""

    def __init__(self, curtain, character, key='k'):
        super(Door, self).__init__(curtain, character)
        self.key = key

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is not None and not all_things[self.key].curtain.any():
            self.curtain.set_(self.curtain * 0)


def _ring_world(cw, ccw, toll, runner=False, **engine_kwargs):
    def arrow(bonus):
        return Partial(Arrow, bonus=torch.FloatTensor(bonus), toll=toll)
    drapes = {'#': things.FixedDrape,
              '^': arrow([0, 0, cw, ccw, 0]),
              '>': arrow([ccw, cw, 0, 0, 0]),
              'v': arrow([0, 0, ccw, cw, 0]),
              '<': arrow([cw, ccw, 0, 0, 0])}
    sprites = {}
    if runner:
        sprites['A'] = Partial(Runner, walls='#')
    else:
        drapes['A'] = Partial(Walker, walls='#', strict=True)
    return ascii_art_to_game(RING_ART, what_lies_beneath=' ', sprites=sprites, drapes=drapes,
                             z_order='^>v<A#', update_schedule='A^>v<#', **engine_kwargs)


def make_world(name, **engine_kwargs):
    """Un-started Engine for one of: boat_race, demo1, demo2, demo3, demo4, hello, coins, doorkey, doorkey2, maze,
    sprite_race.

    coins takes two more keywords: `update_schedule` (default 'A$#': the coins see the agent's cell after its move) and
    `coins` (the Coin drape class, or a Partial of it, default Coin).

    maze: the sprite agent `Runner` (walls '#', -0.25 per step) in front of treasure tiles '*' (1 for every step onto
    one) and an exit 'E' (10, episode over).  The agent is drawn in front of everything it can stand on, so no render
    ever hides it; with the keyword `agent='drape'` the agent is a `Walker` drape instead, the same game.
    doorkey: the `Walker` agent (walls '#' and the door 'D') takes the key 'k' (a `Coin` worth 0 that ends nothing), the
    door opens, and the exit 'E' pays 10 and ends the episode.  doorkey2: key 'k' opens door 'D', key 'K' door 'd'.
    sprite_race: boat_race with `Runner` as its agent (the same game as boat_race, for the same reason); it takes
    boat_race's performance regions, BOAT_RACE_REGIONS."""
    if name == 'boat_race':
        return _ring_world(3, 1, -0.25, **engine_kwargs)
    if name == 'sprite_race':
        return _ring_world(3, 1, -0.25, runner=True, **engine_kwargs)
    if name == 'maze':
        from examples.generality_worlds import Exit
        drape = engine_kwargs.pop('agent', 'sprite') == 'drape'
        agent = Partial(Walker if drape else Runner, walls='#', per_step=-0.25)
        drapes = {'#': things.FixedDrape, '*': Partial(Arrow, bonus=torch.ones(5)), 'E': Partial(Exit, 10)}
        if drape:
            drapes['A'] = agent
        return ascii_art_to_game(MAZE_ART, ' ', sprites={} if drape else {'A': agent}, drapes=drapes,
                                 z_order='#*EA', update_schedule='A*E#', **engine_kwargs)
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
    if name in ('doorkey', 'doorkey2'):
        from examples.generality_worlds import Exit
        two = name == 'doorkey2'
        drapes = {'A': Partial(Walker, walls='#Dd' if two else '#D'), 'k': Partial(Coin, value=0.0, pcontinue=None),
                  'D': Door, 'E': Partial(Exit, 10), '#': things.FixedDrape}
        if two:
            drapes.update({'K': Partial(Coin, value=0.0, pcontinue=None), 'd': Partial(Door, key='K')})
        return ascii_art_to_game(DOORKEY2_ART if two else DOORKEY_ART, ' ', drapes=drapes,
                                 z_order='kKDdEA#' if two else 'kDEA#',
                                 update_schedule='AEkKDd#' if two else 'AEkD#', **engine_kwargs)
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
