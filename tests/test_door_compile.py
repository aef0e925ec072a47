"""The compiler's fit of key-locked door drapes (CX_KIND_DOOR), its refusals, and a pickup world unchanged by the probes
doors brought.  Host only: no GPU."""
import ctypes
import hashlib

import numpy as np
import pytest

from campx_b200 import _native as N
from campx_b200 import things
from campx_b200.ascii_art import Partial, ascii_art_to_game
from campx_b200.compiler import CompileError
from campx_b200.engine import Engine
from examples.generality_worlds import Exit
from examples.worlds import DOORKEY_ART, Coin, Door, Walker, make_world

KEY = Partial(Coin, value=0.0, pcontinue=None)


class PayingDoor(Door):
    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        was = bool(self.curtain.any())
        super(PayingDoor, self).update(actions, board, layers, backdrop, all_things, the_plot)
        if was and not self.curtain.any():
            the_plot.add_reward(1.0)


class TwoKeyDoor(Door):
    """Opens once both 'k' and 'K' are taken."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is not None and not all_things['k'].curtain.any() and not all_things['K'].curtain.any():
            self.curtain.set_(self.curtain * 0)


class HalfDoor(Door):
    """Clears only its first row once the key is taken."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is not None and not all_things[self.key].curtain.any():
            keep = self.curtain.clone()
            keep[1, :] = 0
            self.curtain.set_(self.curtain * (1 - keep))


def _game(art=DOORKEY_ART, z_order='kDEA#', schedule='AEkD#', drapes=None, **kw):
    d = {'A': Partial(Walker, walls='#D'), 'k': KEY, 'D': Door, 'E': Partial(Exit, 10), '#': things.FixedDrape}
    d.update(drapes or {})
    return ascii_art_to_game(art, ' ', drapes=d, z_order=z_order, update_schedule=schedule, **kw)


def _entities(spec):
    return {e.character: e for e in spec.entities}


def test_doorkey_fits_a_door():
    spec = make_world('doorkey').compile()
    ents = _entities(spec)
    assert ents['D'].kind == N.CX_KIND_DOOR and ents['D'].door_key == 'k'
    assert ents['D'].summary() == {"char": "D", "kind": "door", "rank": 3, "group": 0, "door_key": "k"}
    assert ents['k'].kind == N.CX_KIND_PICKUP and ents['k'].terminate_emptied is None
    assert ents['A'].blockers == '#D'
    # the exit lies behind the door: only the probes with the key taken reach it
    assert ents['E'].terminate_on == {1: {'E': 0.0}, 3: {'E': 0.0}}
    d, _ = spec.to_ctypes()
    z = [e.character for e in spec.entities]
    assert d.entities[z.index('D')].kind == N.CX_KIND_DOOR and d.entities[z.index('D')].door_key == z.index('k')


def test_two_keys_two_doors_fit():
    spec = make_world('doorkey2').compile()
    ents = _entities(spec)
    assert (ents['D'].kind, ents['D'].door_key, ents['d'].kind, ents['d'].door_key) == \
        (N.CX_KIND_DOOR, 'k', N.CX_KIND_DOOR, 'K')
    assert ents['K'].kind == N.CX_KIND_PICKUP          # found behind the first door
    assert 2 in ents['E'].terminate_on                 # the exit is reached from above: behind both doors


def test_the_issue_worlds():
    # the door updates before its key: it would open a step late.  Before doors, this compiled with 'D' static.
    with pytest.raises(CompileError, match=r"door drape 'D' updates before its key drape 'k'"):
        _game(schedule='ADkE#').compile()
    assert _entities(_game(schedule='AkDE#').compile())['D'].kind == N.CX_KIND_DOOR


def test_refuses_a_door_opened_by_two_drapes():
    art = ['#########', '#A  #   #', '# K D   #', '# k #  E#', '#########']
    with pytest.raises(CompileError, match=r"drape 'D' changes its curtain in a way that is neither static, a pickup "
                                           r"nor a door"):
        _game(art, z_order='kKDEA#', schedule='AEkKD#', drapes={'K': KEY, 'D': TwoKeyDoor}).compile()


def test_refuses_a_door_that_pays():
    with pytest.raises(CompileError, match=r"door drape 'D' calls \['reward'\]"):
        _game(drapes={'D': PayingDoor}).compile()


def test_refuses_a_door_that_only_partly_clears():
    art = ['#########', '#A  D   #', '#   D   #', '# k #  E#', '#########']
    with pytest.raises(CompileError, match=r"drape 'D' changes its curtain in a way that is neither static, a pickup "
                                           r"nor a door"):
        _game(art, drapes={'D': HalfDoor}).compile()


def _prefilled(door_cells):
    grid = np.array([list(r) for r in DOORKEY_ART])
    door = np.zeros(grid.shape, bool)
    for r, c in door_cells:
        door[r, c] = True
    e = Engine(*grid.shape)
    e.add_prefilled_drape('A', grid == 'A', Walker, walls='#')      # the door does not stop the agent here
    e.add_prefilled_drape('k', grid == 'k', Coin, value=0.0, pcontinue=None)
    e.add_prefilled_drape('D', door, Door)
    e.add_prefilled_drape('#', grid == '#', things.FixedDrape)
    e.set_z_order('kDA#')
    e.set_prefilled_backdrop(' ', np.full(grid.shape, ord(' ')), things.Backdrop)
    return e


def test_refuses_a_door_on_an_item_or_on_the_agents_start():
    with pytest.raises(CompileError, match=r"door drape 'D' shares a cell with an item of pickup drape 'k'"):
        _prefilled([(2, 4), (3, 2)]).compile()
    with pytest.raises(CompileError, match=r"door drape 'D' covers the agent's initial cell"):
        _prefilled([(2, 4), (1, 1)]).compile()


def test_refuses_a_door_in_front_of_the_agent():
    with pytest.raises(CompileError, match=r"door drape 'D' lies in front of the agent 'A'"):
        _game(z_order='kEAD#').compile()


def test_refuses_four_doors():
    art = ['##########', '#A  D d  #', '#   F f E#', '# k ######', '##########']
    drapes = {'A': Partial(Walker, walls='#DdFf')}
    drapes.update({c: Door for c in 'DdFf'})
    with pytest.raises(CompileError, match=r"more than 3 door drapes \(door drape 'f'\)"):
        _game(art, z_order='kDdFfEA#', schedule='AEkDdFf#', drapes=drapes).compile()


# sha256 of the GameDesc content (entities up to the pickup fields, pointers excluded) of the coins world, recorded with
# the compiler before doors existed: the probes with emptied pickup drapes change nothing for it.
PARENT_DIGESTS = {
    'A$#': '6a1841b2cfcd1f1f211057c4b938c21bc641cb178990ed686e09a20a5c58ab05',
    '$A#': 'dc464ffd6d1f843b7d893e482d48f2dba6f74040449f16a06bf73a2e4609210c',
}


def _digest(spec):
    d, keep = spec.to_ctypes()
    h = hashlib.sha256()
    end = N.EntityDesc.emptied_value.offset + N.EntityDesc.emptied_value.size
    for z in range(d.n_entities):
        h.update(ctypes.string_at(ctypes.addressof(d.entities[z]), end))
    for name, _ in N.GameDesc._fields_:
        if name not in ("abi_version", "entities", "backdrop", "masks", "perf_regions"):
            f = getattr(N.GameDesc, name)
            h.update(ctypes.string_at(ctypes.addressof(d) + f.offset, f.size))
    for k in keep:
        if k is not None:
            h.update(k.tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("schedule", sorted(PARENT_DIGESTS))
def test_coins_compiles_to_the_same_bytes(schedule):
    spec = make_world('coins', update_schedule=schedule).compile()
    assert all(e.kind != N.CX_KIND_DOOR for e in spec.entities)
    assert _digest(spec) == PARENT_DIGESTS[schedule]
