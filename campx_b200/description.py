"""Primitive-level description of a game: what the game compiler (campx_b200/compiler) produces at
`Engine.its_showtime()` and what `cx_game_create` consumes (include/campx_b200.h `cx_game_desc`).

One `EntitySpec` per Sprite/Drape in z-order (back to front, campx/engine.py:406-430).  All
per-action lists are indexed by the discrete action index.
"""
import ctypes
import dataclasses
from typing import Dict, List, Optional

import numpy as np

from . import _native as N

KIND_NAMES = {N.CX_KIND_STATIC: "static", N.CX_KIND_CELL: "cell", N.CX_KIND_ROLL: "roll",
              N.CX_KIND_SPRITE: "sprite", N.CX_KIND_PICKUP: "pickup"}


@dataclasses.dataclass
class EntitySpec:
    character: str
    kind: int
    mask: np.ndarray                      # uint8 [rows, cols] curtain after its_showtime (drapes)
    update_rank: int
    update_group: int = 0
    visible: bool = True
    init_pos: Optional[tuple] = None      # sprites: (row, col) after its_showtime
    moves: Optional[List[tuple]] = None   # per action (d_row, d_col), toroidal
    blockers: str = ""                    # characters that refuse a CELL move
    step_reward: Optional[List[Optional[float]]] = None   # per action; None = add_reward not called
    watch: Optional[str] = None           # character of the watched CELL/SPRITE entity
    entry_reward: Optional[Dict[int, Dict[str, float]]] = None   # action -> {char seen: extra reward}
    terminate: Optional[Dict[int, float]] = None          # action -> discount passed to terminate_episode
    terminate_on: Optional[Dict[int, Dict[str, float]]] = None   # action -> {char seen under `watch`: discount}:
                                                          # terminate_episode called only there ("reach the goal")
    discount: Optional[Dict[int, float]] = None           # action -> change_default_discount value
    visible_op: Optional[List[int]] = None                # sprites, per action: CX_VIS_* applied to Sprite.visible
    z_orders: Optional[Dict[int, List[tuple]]] = None     # action -> [(move_this, in_front_of_that or None), ...]
    terminate_emptied: Optional[float] = None             # pickups: discount passed to terminate_episode by the step
                                                          # that takes the last item (None: no such call)

    def summary(self):
        out = {"char": self.character, "kind": KIND_NAMES[self.kind], "rank": self.update_rank,
               "group": self.update_group}
        if self.kind not in (N.CX_KIND_STATIC, N.CX_KIND_PICKUP):
            out["moves"] = [tuple(m) for m in (self.moves or [])]
        if self.blockers:
            out["blockers"] = "".join(sorted(self.blockers))
        if self.step_reward is not None and any(r is not None for r in self.step_reward):
            out["step_reward"] = list(self.step_reward)
        if self.watch is not None:
            out["watch"] = self.watch
            out["entry_reward"] = {a: dict(sorted(v.items())) for a, v in sorted((self.entry_reward or {}).items()) if v}
        if self.terminate:
            out["terminate"] = dict(self.terminate)
        if self.terminate_on:
            out["watch"] = self.watch
            out["terminate_on"] = {a: dict(sorted(v.items())) for a, v in sorted(self.terminate_on.items())}
        if self.discount:
            out["discount"] = dict(self.discount)
        if self.kind == N.CX_KIND_SPRITE:
            out["init_pos"] = tuple(self.init_pos)
            out["visible"] = bool(self.visible)
        if self.visible_op and any(self.visible_op):
            out["visible_op"] = [("keep", "show", "hide", "toggle")[v] for v in self.visible_op]
        if self.z_orders:
            out["z_orders"] = {a: list(v) for a, v in sorted(self.z_orders.items())}
        if self.terminate_emptied is not None:
            out["terminate_emptied"] = self.terminate_emptied
        return out


@dataclasses.dataclass
class GameSpec:
    rows: int
    cols: int
    chars: str                            # every character the renderer knows, sorted by code point
    n_actions: int
    entities: List[EntitySpec]            # z-order, back to front
    backdrop: np.ndarray                  # uint8 [rows, cols] Backdrop.curtain after its_showtime
    n_groups: int = 1
    max_episode_steps: int = 0
    auto_reset: bool = True
    track_returns: bool = False
    first_reward: Optional[float] = None
    first_discount: float = 1.0
    action_format: str = "index"          # how the world's update() methods take actions (host side only)
    backdrop_moves: Optional[List[tuple]] = None   # per action (d_row, d_col): Backdrop.update() rolls its curtain
    occlusion_in_layers: bool = True      # False: unoccluded layers (engine.py:31, rendering.py:227-353)
    performance_regions: Optional[np.ndarray] = None   # uint8 [rows, cols] safety-performance regions (1..R clockwise)

    def summary(self):
        return {"rows": self.rows, "cols": self.cols, "chars": self.chars, "n_actions": self.n_actions,
                "n_groups": self.n_groups, "action_format": self.action_format,
                "first_reward": self.first_reward, "first_discount": self.first_discount,
                **({"backdrop_moves": [tuple(m) for m in self.backdrop_moves]}
                   if self.backdrop_moves and any(m != (0, 0) for m in self.backdrop_moves) else {}),
                "entities": [e.summary() for e in self.entities]}

    def validate(self):
        if sorted(set(self.chars)) != list(self.chars):
            raise ValueError("GameSpec.chars must be sorted and unique")
        if len(self.chars) > N.CX_MAX_CHARS:
            raise NotImplementedError("more than %d distinct characters" % N.CX_MAX_CHARS)
        if len(self.entities) > N.CX_MAX_ENTITIES:
            raise NotImplementedError("more than %d sprites and drapes" % N.CX_MAX_ENTITIES)
        if not 1 <= self.n_actions <= N.CX_MAX_ACTIONS:
            raise NotImplementedError("n_actions must be in 1..%d" % N.CX_MAX_ACTIONS)
        if self.rows * self.cols > N.CX_MAX_CELLS or self.rows > 255 or self.cols > 255:
            raise NotImplementedError("board larger than %d cells" % N.CX_MAX_CELLS)

    def to_ctypes(self):
        """-> (GameDesc, keepalive) ; keepalive holds the numpy buffers the struct points into."""
        self.validate()
        d = N.GameDesc()
        d.abi_version = N.CX_ABI_VERSION
        d.rows, d.cols = self.rows, self.cols
        d.n_chars = len(self.chars)
        for k, ch in enumerate(self.chars):
            d.chars[k] = ord(ch)
        d.n_actions = self.n_actions
        d.n_entities = len(self.entities)
        d.n_groups = self.n_groups
        cells = self.rows * self.cols
        z_of = {e.character: z for z, e in enumerate(self.entities)}
        masks = np.zeros((max(1, len(self.entities)), cells), dtype=np.uint8)
        for z, e in enumerate(self.entities):
            c = d.entities[z]
            c.character = ord(e.character)
            c.kind = e.kind
            c.visible = 1 if e.visible else 0
            c.update_group = e.update_group
            c.update_rank = e.update_rank
            if e.init_pos is not None:
                c.init_row, c.init_col = int(e.init_pos[0]), int(e.init_pos[1])
            masks[z] = np.asarray(e.mask, dtype=np.uint8).reshape(-1) != 0
            moves = e.moves or [(0, 0)] * self.n_actions
            for a in range(self.n_actions):
                c.move_dr[a], c.move_dc[a] = int(moves[a][0]), int(moves[a][1])
            bl = 0
            for ch in e.blockers:
                if ch in self.chars:
                    bl |= 1 << self.chars.index(ch)
            c.blockers = bl
            c.watch = -1 if e.watch is None else z_of[e.watch]
            ra = ta = da = 0
            for a in range(self.n_actions):
                sr = None if e.step_reward is None else e.step_reward[a]
                if sr is not None:
                    ra |= 1 << a
                    c.step_reward[a] = float(sr)
                for ch, v in ((e.entry_reward or {}).get(a) or {}).items():
                    c.entry_reward[a][self.chars.index(ch)] = float(v)
                if e.discount and a in e.discount:
                    da |= 1 << a
                    c.discount_value[a] = float(e.discount[a])
                if e.terminate and a in e.terminate:
                    ta |= 1 << a
                    c.discount_value[a] = float(e.terminate[a])
            c.reward_actions, c.terminate_actions, c.discount_actions = ra, ta, da
            for a, table in (e.terminate_on or {}).items():
                values = set(table.values())
                if len(values) != 1:
                    raise NotImplementedError("terminate_episode discounts that depend on the character reached")
                c.terminate_value[a] = float(values.pop())
                bits = 0
                for ch in table:
                    bits |= 1 << self.chars.index(ch)
                c.terminate_chars[a] = bits
            for a in range(self.n_actions):
                c.visible_op[a] = int(e.visible_op[a]) if e.visible_op else N.CX_VIS_KEEP
                zd = (e.z_orders or {}).get(a) or []
                if len(zd) > N.CX_MAX_ZDIRS:
                    raise NotImplementedError("more than %d change_z_order calls by one entity in one step"
                                              % N.CX_MAX_ZDIRS)
                c.n_zdirs[a] = len(zd)
                for k, (move_this, front_of) in enumerate(zd):
                    c.z_move[a][k] = z_of[move_this]
                    c.z_front[a][k] = -1 if front_of is None else z_of[front_of]
            if e.terminate_emptied is not None:
                c.terminate_emptied, c.emptied_value = 1, float(e.terminate_emptied)
        backdrop = np.ascontiguousarray(np.asarray(self.backdrop, dtype=np.uint8).reshape(-1))
        masks = np.ascontiguousarray(masks)
        d.backdrop = backdrop.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
        d.masks = masks.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
        d.max_episode_steps = int(self.max_episode_steps)
        d.auto_reset = 1 if self.auto_reset else 0
        d.track_returns = 1 if self.track_returns else 0
        d.first_reward = float("nan") if self.first_reward is None else float(self.first_reward)
        d.first_discount = float(self.first_discount)
        for a, (dr, dc) in enumerate(self.backdrop_moves or []):
            d.backdrop_dr[a], d.backdrop_dc[a] = int(dr), int(dc)
        d.unoccluded_layers = 0 if self.occlusion_in_layers else 1
        regions = None
        if self.performance_regions is not None:
            regions = np.ascontiguousarray(np.asarray(self.performance_regions, dtype=np.uint8).reshape(-1))
            d.perf_regions = regions.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
            d.n_perf_regions = int(regions.max())
        return d, (backdrop, masks, regions)
