"""TEST INFRASTRUCTURE ONLY -- the oracle of games with key-locked doors (CX_KIND_DOOR drapes).

It extends the pickup oracle (tests/helpers/pickup_oracle.py) with the door rule, restated mask-level and single-env on
the numpy oracle of oracle/campx_oracle.py: `KeyDrape` is a collectible item that pays nothing and ends nothing, and
`DoorDrape` clears its whole curtain in the first step that finds its key drape empty.  `doorkey_world` is
examples/worlds.py's `doorkey` (or `doorkey2`) built from them, the oracle's boat_race agent with the door among its
walls, and the oracle's exit.

Parity status: UNPINNED BY THE REFERENCE, like pickups.  The reference ships no world with doors; what the kernels are
held to is this restatement and, at compile time, the user's own classes on the compiler's shadow.
"""
import numpy as np

from examples.worlds import DOORKEY_ART, DOORKEY2_ART
from oracle import campx_oracle as O
from tests.helpers.pickup_oracle import (CX_FLAG_ALREADY_OVER, CX_FLAG_BAD_ACTION, CX_FLAG_REWARD_NONE,
                                         CX_FLAG_TERMINATED, CX_FLAG_TRUNCATED, N_ACTIONS, PickupDrape)


class KeyDrape(PickupDrape):
    def update(self, actions, board, layers, backdrop, things, the_plot):
        if actions is None:
            return
        here = np.asarray(things['A'].curtain).astype(np.int64)
        if int((self.curtain.astype(np.int64) * here).sum()):
            self.curtain[...] = self.curtain * (1 - here)
            the_plot.add_reward(self.value)


class DoorDrape(O.Drape):
    def __init__(self, curtain, character, key='k'):
        super().__init__(curtain, character)
        self.key = key

    def update(self, actions, board, layers, backdrop, things, the_plot):
        if actions is not None and not np.asarray(things[self.key].curtain).any():
            self.curtain[...] = 0


def doorkey_world(two=False, art=None):
    art = art or (DOORKEY2_ART if two else DOORKEY_ART)
    drapes = {'A': (O.AgentDrape, (), dict(variant='boat_race', blocking_chars='#Dd' if two else '#D')),
              'k': (KeyDrape, (), dict(value=0.0)), 'D': DoorDrape, 'E': (O.ExitDrape, (), dict(prize=10.0)),
              '#': O.FixedDrape}
    if two:
        drapes.update({'K': (KeyDrape, (), dict(value=0.0)), 'd': (DoorDrape, (), dict(key='K'))})
    game = O.ascii_art_to_game(art, ' ', drapes=drapes, z_order='kKDdEA#' if two else 'kDEA#',
                               update_schedule='AEkKDd#' if two else 'AEkD#')
    obs, _, _ = game.its_showtime()
    return game, obs


def items_of(game, two=False, art=None):
    """bit i = item i still on the board: the keys' cells, key drape by key drape in z-order, row-major"""
    art = O.ascii_art_to_array(art or (DOORKEY2_ART if two else DOORKEY_ART)).reshape(-1)
    bits, i = 0, 0
    for key in ('k', 'K') if two else ('k',):
        cur = np.asarray(game.things[key].curtain).reshape(-1)
        for c in np.flatnonzero(art == ord(key)):
            bits |= int(bool(cur[c])) << i
            i += 1
    return bits


def rollout(actions, two=False, limit=0, auto_reset=True, art=None):
    """One env: per action index yield (board uint8 [R, C], layered uint8 [L, R, C], reward f32, discount f32, flags,
    items) as the batched engine reports them (see pickup_oracle.rollout)."""
    game, obs = doorkey_world(two, art)
    every = items_of(game, two, art)
    frame, steps, over = obs, 0, False
    for a in actions:
        a = int(a)
        if over or a >= N_ACTIONS:
            yield (np.asarray(frame.board).astype(np.uint8), np.asarray(frame.layered_board).astype(np.uint8),
                   0.0, 0.0 if over else 1.0,
                   (CX_FLAG_ALREADY_OVER if over else CX_FLAG_BAD_ACTION) | CX_FLAG_REWARD_NONE, items_of(game, two, art))
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
        done = flags & (CX_FLAG_TERMINATED | CX_FLAG_TRUNCATED)
        yield (np.asarray(frame.board).astype(np.uint8), np.asarray(frame.layered_board).astype(np.uint8),
               float(np.float32(0.0 if reward is None else reward)), float(np.float32(discount)), flags,
               every if (auto_reset and done) else items_of(game, two, art))
        if done:
            if auto_reset:
                game, frame = doorkey_world(two, art)
                steps = 0
            else:
                over = True
