"""Build an `Engine` from ASCII art: the construction side of the drop-in boundary.

Same entry points as `campx/ascii_art.py`: `ascii_art_to_long_tensor` (:29-57),
`ascii_art_to_game` (:60-309) and `Partial` (:311-340), with the same argument meaning, defaults,
validation and exception classes.  Extra keyword arguments (`num_envs`, `device`, `num_actions`,
`action_format`, `max_episode_steps`, `auto_reset`, `track_returns`, `performance_regions`, `verify`) are forwarded to
`Engine` -- they are the only additions.
"""
import itertools

import numpy as np
import torch

from . import things
from .engine import Engine


def ascii_art_to_long_tensor(art):
    """List/tuple of equal-length ASCII strings -> int64 [rows, cols] tensor of character codes."""
    message = ('the argument to ascii_art_to_long_tensor must be a list (or tuple) of strings containing '
               'the same number of strictly-ASCII characters.')
    if not isinstance(art, (list, tuple)) or not all(isinstance(row, str) for row in art):
        raise TypeError(message + ' Did you pass a list of list of single characters?')
    if not art or len(set(len(row) for row in art)) != 1:
        raise ValueError(message)
    try:
        rows = [np.frombuffer(row.encode('ascii'), dtype=np.uint8) for row in art]
    except UnicodeEncodeError:
        raise ValueError(message)
    return torch.from_numpy(np.vstack(rows).astype(np.int64))


class Partial(object):
    """A Backdrop/Sprite/Drape subclass together with its extra constructor arguments."""

    def __init__(self, pycolab_thing, *args, **kwargs):
        if not issubclass(pycolab_thing, (things.Backdrop, things.Sprite, things.Drape)):
            raise TypeError('the pycolab_thing argument to ascii_art.Partial must be a Backdrop, Sprite, or '
                            'Drape subclass.')
        self.pycolab_thing = pycolab_thing
        self.args = args
        self.kwargs = kwargs


def _as_partial(thing):
    return thing if isinstance(thing, Partial) else Partial(thing)


def ascii_art_to_game(art, what_lies_beneath, sprites=None, drapes=None, backdrop=things.Backdrop,
                      update_schedule=None, z_order=None, occlusion_in_layers=True, **engine_kwargs):
    """Construct an `Engine` whose sprites, drapes and backdrop are read off an ASCII-art diagram.

    art: list of strings; every character that is a key of `sprites`/`drapes` becomes that entity's
        initial position/mask and is replaced in the backdrop by `what_lies_beneath` (a single
        character or art of the same shape).
    update_schedule: order in which entities are consulted each step; a flat list/string is ONE update
        group, a list of lists is several (the board is re-rendered between groups).  Defaults to all
        entity characters in sorted order (the reference's default is `list(set(...))`, i.e. hash order,
        ascii_art.py:178).
    z_order: back-to-front paint order; defaults to the flattened update schedule.
    """
    sprites = {ch: _as_partial(v) for ch, v in (sprites or {}).items()}
    drapes = {ch: _as_partial(v) for ch, v in (drapes or {}).items()}
    backdrop = _as_partial(backdrop)
    entity_chars = set(sprites) | set(drapes)

    if update_schedule is None:
        update_schedule = sorted(entity_chars)
    if isinstance(update_schedule, str):
        update_schedule = list(update_schedule)
    if all(isinstance(item, str) for item in update_schedule):
        update_schedule = [update_schedule]
    try:
        flat_schedule = list(itertools.chain.from_iterable(update_schedule))
    except TypeError:
        raise TypeError('if any element in update_schedule is an iterable (like a list), all elements in '
                        'update_schedule must be')
    if set(flat_schedule) != entity_chars or len(flat_schedule) != len(entity_chars):
        raise ValueError('if specified, update_schedule must list each sprite and drape exactly once.')
    if z_order is None:
        z_order = flat_schedule
    if set(z_order) != entity_chars or len(z_order) != len(entity_chars):
        raise ValueError('if specified, z_order must list each sprite and drape exactly once.')
    if isinstance(what_lies_beneath, str) and len(what_lies_beneath) != 1:
        raise ValueError('what_lies_beneath may either be a single-character ASCII string or a list of '
                         'ASCII-character strings')
    for ch in itertools.chain(entity_chars, ''.join(what_lies_beneath)):
        if not isinstance(ch, str) or len(ch) != 1 or ord(ch) > 127:
            raise ValueError('keys of sprites, keys of drapes, what_lies_beneath (or its entries), values in '
                             'z_order, and (possibly nested) values in update_schedule must all be '
                             'single-character ASCII strings.')
    if entity_chars.intersection(''.join(what_lies_beneath)):
        raise ValueError('any character specified in what_lies_beneath must not be one of the characters used '
                         'as keys in the sprites or drapes arguments.')

    art = ascii_art_to_long_tensor(art)
    if isinstance(what_lies_beneath, str):
        beneath = torch.full_like(art, ord(what_lies_beneath))
    else:
        beneath = ascii_art_to_long_tensor(what_lies_beneath)
        if art.shape != beneath.shape:
            raise ValueError('if not a single ASCII character, what_lies_beneath must be ASCII art whose shape '
                             'is the same as that of the ASCII art in art.')

    group_id = {}
    for i, group in enumerate(update_schedule):
        for ch in group:
            group_id[ch] = '{:05d}'.format(i)

    game = Engine(art.shape[0], art.shape[1], occlusion_in_layers=occlusion_in_layers, **engine_kwargs)
    for ch in flat_schedule:
        game.update_group(group_id[ch])
        mask = art == ord(ch)
        if ch in drapes:
            p = drapes[ch]
            game.add_prefilled_drape(ch, mask, p.pycolab_thing, *p.args, **p.kwargs)
        if ch in sprites:
            where = mask.nonzero()
            if len(where) > 1:
                raise ValueError('sprite character {} can appear in at most one place in art.'.format(ch))
            position = (int(where[0][0]), int(where[0][1])) if len(where) else (0, 0)
            p = sprites[ch]
            game.add_sprite(ch, position, p.pycolab_thing, *p.args, **p.kwargs)
        art = torch.where(mask, beneath, art)
    game.set_z_order(z_order)
    palette = ''.join(chr(int(c)) for c in torch.unique(art).tolist())
    game.set_prefilled_backdrop(palette, art, backdrop.pycolab_thing, *backdrop.args, **backdrop.kwargs)
    return game
