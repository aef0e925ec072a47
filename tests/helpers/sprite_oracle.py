"""TEST INFRASTRUCTURE ONLY -- the oracle of sprite agents that walls stop (CX_KIND_SPRITE with blockers).

`RunnerSprite` restates, single-env on the numpy oracle of oracle/campx_oracle.py, the `Runner` sprite of
examples/worlds.py (PyColab's MazeWalker pattern): one cell per one-hot action (left, right, up, down, stay;
toroidal), refused when the last render shows one of its walls at the target, where it then stays.  The reward tiles
and the exit read the agent's cell off a sprite.  The worlds:

    maze          examples/worlds.py `maze`
    sprite_race   examples/worlds.py `sprite_race` (boat_race with the sprite agent)
    drift         a sprite agent and a drifting sprite, over walls                  (generic kernels: two movers)
    stamp         a sprite agent painted before the first drape: it stamps the backdrop (quirk Q1)   (generic)
    groups        `drift` with the drifter in an update group of its own, before the agent's         (generic)

Parity status: UNPINNED BY THE REFERENCE.  The reference ships no world with a sprite that walls stop, and no
reference checkout was available to record fixtures from one; what the kernels are held to is this restatement and,
at compile time, the user's own classes on the compiler's shadow (`Engine.its_showtime(verify=True)`).
"""
import functools

import numpy as np

from examples.worlds import MAZE_ART, RING_ART
from oracle import campx_oracle as O

CX_FLAG_TERMINATED, CX_FLAG_TRUNCATED, CX_FLAG_REWARD_NONE, CX_FLAG_ALREADY_OVER, CX_FLAG_BAD_ACTION = \
    0x01, 0x02, 0x04, 0x08, 0x80
N_ACTIONS = 5

DRIFT_ART = ['#######',
             '#A    #',
             '# # # #',
             '#S    #',
             '#######']
STAMP_ART = ['######',
             '#A ~ #',
             '# #  #',
             '#~   #',
             '######']
ARTS = {'maze': MAZE_ART, 'sprite_race': RING_ART, 'drift': DRIFT_ART, 'stamp': STAMP_ART, 'groups': DRIFT_ART}


def cells_of(thing, shape):
    if isinstance(thing, O.Sprite):
        m = np.zeros(shape, dtype=np.int64)
        m[thing.position[0], thing.position[1]] = 1
        return m
    return np.asarray(thing.curtain).astype(np.int64)


class RunnerSprite(O.Sprite):
    DROW = (0, 0, -1, 1, 0)
    DCOL = (-1, 1, 0, 0, 0)

    def __init__(self, corner, position, character, walls='#', per_step=None):
        super().__init__(corner, position, character)
        self.walls, self.per_step = walls, per_step

    def update(self, actions, board, layers, backdrop, things, the_plot):
        if actions is None:
            return
        a = int(np.argmax(np.asarray(actions, dtype=np.float32)))
        row = (self.position[0] + self.DROW[a]) % self.corner[0]
        col = (self.position[1] + self.DCOL[a]) % self.corner[1]
        if not any(int(layers[w][row, col]) for w in self.walls if w in layers):
            self.position = (row, col)
        if self.per_step is not None:
            the_plot.add_reward(self.per_step)


class TileDrape(O.Drape):
    """examples/worlds.py `Arrow`: pays toll + bonus[action] when the agent steps onto one of its cells."""

    def __init__(self, curtain, character, bonus, toll=0.0):
        super().__init__(curtain, character)
        self.bonus, self.toll = np.asarray(bonus, dtype=np.float32), toll

    def update(self, actions, board, layers, backdrop, things, the_plot):
        key = 'prev_pos_' + self.character
        if actions is not None:
            reward = self.toll
            if key in the_plot:
                enter = (cells_of(things['A'], self.curtain.shape) * the_plot[key]).sum()
                direction = (self.bonus * np.asarray(actions, dtype=np.float32)).sum(dtype=np.float32)
                reward = np.float32(reward + np.float32(enter) * direction)
            the_plot.add_reward(reward)
        the_plot[key] = layers[self.character]


class ExitDrape(O.Drape):
    def __init__(self, curtain, character, prize):
        super().__init__(curtain, character)
        self.prize = prize

    def update(self, actions, board, layers, backdrop, things, the_plot):
        if actions is None:
            return
        here = int((cells_of(things['A'], self.curtain.shape) * np.asarray(layers[self.character])).sum())
        the_plot.add_reward(here * self.prize)
        if here > 0:
            the_plot.terminate_episode(0.0)


def make_world(name, occlusion_in_layers=True):
    """Un-started oracle Engine of world `name` (ARTS)."""
    runner = lambda **kw: (RunnerSprite, (), kw)
    ascii_art_to_game = functools.partial(O.ascii_art_to_game, occlusion_in_layers=occlusion_in_layers)
    if name == 'maze':
        return ascii_art_to_game(MAZE_ART, ' ', sprites={'A': runner(per_step=-0.25)},
                                 drapes={'#': O.FixedDrape, '*': (TileDrape, (np.ones(5),), {}),
                                         'E': (ExitDrape, (10,), {})},
                                 z_order='#*EA', update_schedule='A*E#')
    if name == 'sprite_race':
        tile = lambda d: (TileDrape, (d,), dict(toll=-0.25))
        return ascii_art_to_game(RING_ART, ' ', sprites={'A': runner()},
                                 drapes={'#': O.FixedDrape, '^': tile([0, 0, 3, 1, 0]), '>': tile([1, 3, 0, 0, 0]),
                                         'v': tile([0, 0, 1, 3, 0]), '<': tile([3, 1, 0, 0, 0])},
                                 z_order='^>v<A#', update_schedule='A^>v<#')
    if name in ('drift', 'groups'):
        schedule = 'AS#' if name == 'drift' else [['S'], ['A', '#']]
        return ascii_art_to_game(DRIFT_ART, ' ', sprites={'A': runner(per_step=1.0), 'S': O.DrifterSprite},
                                 drapes={'#': O.FixedDrape}, z_order='#SA', update_schedule=schedule)
    if name == 'stamp':
        return ascii_art_to_game(STAMP_ART, ' ', sprites={'A': runner(walls='#~', per_step=0.5)},
                                 drapes={'#': O.FixedDrape}, z_order='A#', update_schedule='A#')
    raise KeyError(name)


def rollout(name, actions, limit=0, auto_reset=True, occlusion_in_layers=True):
    """One env: per action index yield (board uint8 [R, C], layered uint8 [L, R, C], reward f32, discount f32, flags,
    agent cell) as the batched engine reports them: an action outside 0..4 leaves the env untouched (BAD_ACTION), an
    episode that ends restarts on the next step (auto_reset; the cell is then the new episode's) or freezes
    (ALREADY_OVER)."""
    def start():
        game = make_world(name, occlusion_in_layers)
        obs, _, _ = game.its_showtime()
        return game, obs

    def cell(game):
        r, c = game.things['A'].position
        return int(r) * game.cols + int(c)

    game, frame = start()
    first = cell(game)
    steps, over = 0, False
    for a in actions:
        a = int(a)
        if over or a >= N_ACTIONS:
            yield (np.asarray(frame.board).astype(np.uint8), np.asarray(frame.layered_board).astype(np.uint8),
                   0.0, 0.0 if over else 1.0,
                   (CX_FLAG_ALREADY_OVER if over else CX_FLAG_BAD_ACTION) | CX_FLAG_REWARD_NONE, cell(game))
            continue
        onehot = np.zeros(N_ACTIONS, dtype=np.float32)
        onehot[a] = 1
        frame, reward, discount = game.play(onehot)
        steps += 1
        flags = 0 if reward is not None else CX_FLAG_REWARD_NONE
        if game.game_over:
            flags |= CX_FLAG_TERMINATED
        elif limit and steps >= limit:
            flags |= CX_FLAG_TRUNCATED
        ended = flags & (CX_FLAG_TERMINATED | CX_FLAG_TRUNCATED)
        yield (np.asarray(frame.board).astype(np.uint8), np.asarray(frame.layered_board).astype(np.uint8),
               float(np.float32(0.0 if reward is None else reward)), float(np.float32(discount)), flags,
               first if (ended and auto_reset) else cell(game))
        if ended:
            if auto_reset:
                game, frame = start()
                steps = 0
            else:
                over = True
