"""The compiler's fit of collectible-item drapes (CX_KIND_PICKUP), its refusals, and pickup-free worlds unchanged.
Host only: no GPU."""
import ctypes
import hashlib

import numpy as np
import pytest
import torch

from campx_b200 import _native as N
from campx_b200 import things
from campx_b200.ascii_art import Partial, ascii_art_to_game
from campx_b200.compiler import CompileError
from examples import generality_worlds, worlds
from examples.worlds import Coin, Walker


class Coins(things.Drape):
    """The drape of the issue that asked for pickups, verbatim."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        here = all_things['A'].curtain
        if (self.curtain * here).sum():
            self.curtain.set_(self.curtain * (1 - here))
            the_plot.add_reward(1.0)
            if not self.curtain.any():
                the_plot.terminate_episode()


class CountingCoins(Coins):
    """Pays 1 for the first coin and 2 for every other: depends on more than the action."""

    def update(self, actions, board, layers, backdrop, all_things, the_plot):
        if actions is None:
            return
        here = all_things['A'].curtain
        if (self.curtain * here).sum():
            full = int(self.curtain.sum()) == 3
            self.curtain.set_(self.curtain * (1 - here))
            the_plot.add_reward(1.0 if full else 2.0)


def _game(art, drapes=None, z_order='$A#', schedule='A$#', **kw):
    d = {'A': Partial(Walker, walls='#'), '$': Coins, '#': things.FixedDrape}
    d.update(drapes or {})
    return ascii_art_to_game(art, ' ', drapes=d, z_order=z_order, update_schedule=schedule, **kw)


NEXT_TO_START = ['#######', '#A$ $ #', '# # # #', '#   $ #', '#######']
AWAY_FROM_START = ['#######', '#A  $ #', '# # # #', '#$  $ #', '#######']


@pytest.mark.parametrize("art", [NEXT_TO_START, AWAY_FROM_START])
@pytest.mark.parametrize("schedule", ["A$#", "$A#"])
def test_coin_drape_is_a_pickup(art, schedule):
    spec = _game(art, schedule=schedule).compile()
    coin = {e.character: e for e in spec.entities}['$']
    assert coin.kind == N.CX_KIND_PICKUP
    assert coin.watch == 'A' and coin.terminate_emptied == 0.0
    assert coin.entry_reward == {a: {'$': 1.0} for a in range(5)}
    assert coin.step_reward is None and coin.summary()["kind"] == "pickup"
    d, _ = spec.to_ctypes()
    z = [e.character for e in spec.entities].index('$')
    assert d.entities[z].kind == N.CX_KIND_PICKUP and d.entities[z].terminate_emptied == 1
    assert d.entities[z].entry_reward[0][spec.chars.index('$')] == 1.0


def test_coins_world_and_its_discount():
    spec = worlds.make_world('coins', coins=Partial(Coin, pcontinue=0.25)).compile()
    coin = {e.character: e for e in spec.entities}['$']
    assert coin.kind == N.CX_KIND_PICKUP and coin.terminate_emptied == 0.25
    assert int(np.count_nonzero(coin.mask)) == 10


def _refused(match, **kw):
    with pytest.raises(CompileError, match=match):
        _game(**kw).compile()


def test_refuses_items_above_the_agent():
    _refused(r"pickup drape '\$' lies in front of the agent", art=NEXT_TO_START, z_order='A$#')


def test_refuses_an_item_under_the_agents_start():
    art = ['#####', '#A  #', '#####']
    prefill_coin = np.zeros((3, 5), np.uint8)
    prefill_coin[1, 1] = prefill_coin[1, 3] = 1
    from campx_b200.engine import Engine
    e = Engine(3, 5)
    e.add_prefilled_drape('A', (np.array([list(r) for r in art]) == 'A'), Walker, walls='#')
    e.add_prefilled_drape('$', prefill_coin, Coins)
    e.add_prefilled_drape('#', (np.array([list(r) for r in art]) == '#'), things.FixedDrape)
    e.set_z_order('$A#')
    e.set_prefilled_backdrop(' ', np.full((3, 5), ord(' ')), things.Backdrop)
    with pytest.raises(CompileError, match=r"pickup drape '\$' has an item under the agent's initial cell"):
        e.compile()


def test_refuses_two_pickups_on_one_cell():
    art = ['######', '#A$  #', '######']
    from campx_b200.engine import Engine
    e = Engine(3, 6)
    grid = np.array([list(r) for r in art])
    e.add_prefilled_drape('A', grid == 'A', Walker, walls='#')
    e.add_prefilled_drape('$', grid == '$', Coins)
    e.add_prefilled_drape('%', grid == '$', Coins)
    e.add_prefilled_drape('#', grid == '#', things.FixedDrape)
    e.set_z_order('$%A#')
    e.set_prefilled_backdrop(' ', np.full((3, 6), ord(' ')), things.Backdrop)
    with pytest.raises(CompileError, match=r"pickup drapes '\$' and '%' share cell"):
        e.compile()


def test_refuses_more_than_64_items():
    art = ['#' * 12] + ['#' + ('A' if r == 0 else '$') + '$' * 9 + '#' for r in range(7)] + ['#' * 12]
    _refused(r"more than 64 item cells in all \(pickup drape '\$'\)", art=art)


def test_refuses_performance_regions_and_unoccluded_layers():
    regions = np.zeros((5, 7), np.uint8)
    regions[1, 1], regions[1, 2] = 1, 2
    _refused(r"pickup drape '\$' together with performance_regions", art=NEXT_TO_START, track_returns=True,
             performance_regions=regions)
    _refused(r"pickup drape '\$' needs occluded layers", art=NEXT_TO_START, occlusion_in_layers=False)


def test_refuses_games_on_the_generic_kernels():
    class Slider(things.Sprite):
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            pass
    art = ['#########', '#A$ $#S #', '#########']     # the sprite sits in a pocket the agent cannot reach
    g = ascii_art_to_game(art, ' ', sprites={'S': Slider},
                          drapes={'A': Partial(Walker, walls='#'), '$': Coins, '#': things.FixedDrape},
                          z_order='$AS#', update_schedule='A$S#')
    with pytest.raises(CompileError, match=r"pickup drape '\$' needs a single-agent game"):
        g.compile()


def test_refuses_what_depends_on_an_items_presence():
    # the agent pays for stepping onto an empty floor cell, and a taken coin leaves one behind
    _refused(r"entity 'A' depends on whether an item of pickup drape '\$' is present",
             art=NEXT_TO_START, drapes={'A': Partial(Walker, walls='#', treasures=' ')})


def test_refuses_a_reward_that_is_not_a_function_of_the_action():
    _refused(r"the reward of pickup drape '\$' depends on something other than the action",
             art=['#######', '#A$$$ #', '#######'], drapes={'$': CountingCoins})


# sha256 of the GameDesc content (ABI 6 fields, pointers excluded) of every pickup-free example world, recorded with the
# compiler before pickups existed: these worlds still compile to the very same bytes.
PARENT_DIGESTS = {
    'boat_race': 'f8a5a5495f451d70f9cd2b146e9fecaecacff8c9781dacc2bc1d7abf1ac1feb6',
    'demo1': '8c724e66b208f30478ebc1c17ab195a5583f211f873858350c107ec77bef0313',
    'demo2': 'd437eb5526fa3398ca4df970df9c6344ba43dc866d7cd825014b1740ab4ee328',
    'demo3': 'c7cc2e86f05f4ba53cc633f4cc432bd0c221947094f22103bebb41b67cca609d',
    'demo4': '27ed461700a548dd1d86067278f2e34aecf5e83f8ca99eb92ec2c308f81e238e',
    'hello': 'fa2805607ce64b57de53fddb9d1513506c35cf70d93c23507239815a174bb0df',
    'goal': 'fbbdc2a92ee853533b9cd952932c6aa1c031f051df20807530b2d12c615f6977',
    'goal2': '1b0d155db4a52b34e8fb53a5bf1134702dcc1d16c0a914d9efa24d0baa26d247',
    'zswap': '704f098ae4a1f028d35b1a56eb40a67042745600ac15080e575f6d3ce8f5d85b',
    'ghost': '89142b112dda2c04e74ded460b260558fe6daab51856cf7bb2a10d47f4d84598',
    'scroll': 'e9d9699ff207e2734f33509e2c0972d139221174f482a9bdb4ca9b537c789183',
}


def _digest(spec):
    d, keep = spec.to_ctypes()
    h = hashlib.sha256()
    end = N.EntityDesc.z_front.offset + N.EntityDesc.z_front.size
    for z in range(d.n_entities):
        h.update(ctypes.string_at(ctypes.addressof(d.entities[z]), end))
        assert d.entities[z].terminate_emptied == 0 and d.entities[z].emptied_value == 0.0
    for name, _ in N.GameDesc._fields_:
        if name not in ("abi_version", "entities", "backdrop", "masks", "perf_regions"):
            f = getattr(N.GameDesc, name)
            h.update(ctypes.string_at(ctypes.addressof(d) + f.offset, f.size))
    for k in keep:
        if k is not None:
            h.update(k.tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("name", sorted(PARENT_DIGESTS))
def test_pickup_free_worlds_compile_to_the_same_bytes(name):
    if name in ('boat_race', 'demo1', 'demo2', 'demo3', 'demo4', 'hello'):
        spec = worlds.make_world(name).compile()
    else:
        spec = generality_worlds.make_generality_world(name).compile()
    assert all(e.kind != N.CX_KIND_PICKUP for e in spec.entities)
    assert _digest(spec) == PARENT_DIGESTS[name]
