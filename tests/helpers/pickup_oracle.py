"""TEST INFRASTRUCTURE ONLY -- the oracle of games with collectible items (CX_KIND_PICKUP drapes).

`PickupDrape` restates, mask-level and single-env on the numpy oracle of oracle/campx_oracle.py, the plain CampX
drape a user writes for coins, keys or pellets: when the agent stands on one of its cells as it updates, it clears
that cell, adds a reward and, once empty, terminates the episode.  `coins_world` is examples/worlds.py's `coins`
world built from it and the oracle's boat_race agent (the same wall gate as `Walker(walls='#')`).

Parity status: UNPINNED BY THE REFERENCE.  The reference ships no world with collectible items, and no reference
checkout was available to record fixtures from one; what the kernels are held to is this restatement and, at compile
time, the user's own classes on the compiler's shadow (`Engine.its_showtime(verify=True)`).
"""
import numpy as np

from examples.worlds import COINS_ART
from oracle import campx_oracle as O

CX_FLAG_TERMINATED, CX_FLAG_TRUNCATED, CX_FLAG_REWARD_NONE, CX_FLAG_ALREADY_OVER, CX_FLAG_BAD_ACTION = \
    0x01, 0x02, 0x04, 0x08, 0x80
N_ACTIONS = 5


class PickupDrape(O.Drape):
    def __init__(self, curtain, character, value=1.0, pcontinue=0.0):
        super().__init__(curtain, character)
        self.value, self.pcontinue = value, pcontinue

    def update(self, actions, board, layers, backdrop, things, the_plot):
        if actions is None:
            return
        here = np.asarray(things['A'].curtain).astype(np.int64)
        if int((self.curtain.astype(np.int64) * here).sum()):
            self.curtain[...] = self.curtain * (1 - here)
            the_plot.add_reward(self.value)
            if not self.curtain.any():
                the_plot.terminate_episode(self.pcontinue)


def coins_world(schedule='A$#', pcontinue=0.0, art=COINS_ART):
    game = O.ascii_art_to_game(art, ' ', drapes={'A': (O.AgentDrape, (), dict(variant='boat_race')),
                                                       '$': (PickupDrape, (), dict(pcontinue=pcontinue)),
                                                       '#': O.FixedDrape},
                               z_order='$A#', update_schedule=schedule)
    obs, _, _ = game.its_showtime()
    return game, obs


def items_of(game, art=COINS_ART):
    """bit i = coin i (row-major) still on the board"""
    cur = np.asarray(game.things['$'].curtain).reshape(-1)
    cells = np.flatnonzero(O.ascii_art_to_array(art).reshape(-1) == ord('$'))
    return sum(1 << i for i, c in enumerate(cells) if cur[c])


def rollout(actions, schedule='A$#', limit=0, auto_reset=True, pcontinue=0.0, art=COINS_ART):
    """One env: per action index yield (board uint8 [R, C], layered uint8 [L, R, C], reward f32, discount f32, flags,
    items) as the batched engine reports them: an action outside 0..4 leaves the env untouched (BAD_ACTION), an
    episode that ends restarts on the next step (auto_reset: its items are those of the new episode) or freezes
    (ALREADY_OVER)."""
    game, obs = coins_world(schedule, pcontinue, art)
    frame, steps, over = obs, 0, False
    for a in actions:
        a = int(a)
        if over:
            yield (np.asarray(frame.board).astype(np.uint8), np.asarray(frame.layered_board).astype(np.uint8),
                   0.0, 0.0, CX_FLAG_ALREADY_OVER | CX_FLAG_REWARD_NONE, items_of(game, art))
            continue
        if a >= N_ACTIONS:
            yield (np.asarray(frame.board).astype(np.uint8), np.asarray(frame.layered_board).astype(np.uint8),
                   0.0, 1.0, CX_FLAG_BAD_ACTION | CX_FLAG_REWARD_NONE, items_of(game, art))
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
        yield (np.asarray(frame.board).astype(np.uint8), np.asarray(frame.layered_board).astype(np.uint8),
               float(np.float32(0.0 if reward is None else reward)), float(np.float32(discount)), flags,
               items_of(game, art) if not (auto_reset and flags & (CX_FLAG_TERMINATED | CX_FLAG_TRUNCATED))
               else (1 << len(np.flatnonzero(O.ascii_art_to_array(art) == ord('$')))) - 1)
        if flags & (CX_FLAG_TERMINATED | CX_FLAG_TRUNCATED):
            if auto_reset:
                game, frame = coins_world(schedule, pcontinue, art)
                steps = 0
            else:
                over = True
