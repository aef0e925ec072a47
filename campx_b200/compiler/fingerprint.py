"""Behavioural fingerprinting of user entity classes -> kernel primitives (GameSpec).

Why fingerprinting: CampX game rules are arbitrary Python in `update()` methods written for ONE
[R,C] tensor, with Python control flow on data (`assert sum(act) == 1`, examples/boat_race.py:48;
`if actions == 4`, Hello World notebook cell 3) and numpy round trips (`np.roll(self.curtain.numpy())`)
-- they cannot be traced or vmapped.  Instead each entity is observed on a single-env CPU shadow
(shadow.py) under a set of probes, fitted to a primitive, and the fit is checked on EVERY probe;
anything that does not fit raises `CompileError` (a NotImplementedError): there is no fallback.
Entities that keep state of their own (a step counter, a visited set, an RNG) are detected by comparing
their instance attributes and the Plot's non-tensor entries before and after every probe, and refused.

Probe set
  * every action from the post-its_showtime state;
  * for a one-cell drape ("agent"): every action from every cell reachable by breadth-first search
    over its own observed moves (8 cells for boat_race, 25 for Demo 1);
  * for sprites / rolling drapes: every action from the board corners and a few interior
    positions/offsets (pins the toroidal wrap);
  * for a sprite that walls stop (no fixed displacement from the corners): every action from every position
    reachable by breadth-first search over its own observed moves, as for a one-cell drape.

  * for sprites that change `_visible`: every action from the other visibility state;
  * for a Backdrop whose update() changes its curtain: every action from a few pre-rolled curtains.
  * for a pickup drape (collectible items): every probe above that took an item again with that item already
    taken, and with that item as the drape's last one;
  * for every pickup drape, and for all of them together: the drape emptied, with what that opens open, every action
    from every cell the agent reaches there; and the drape holding one item only (this is what shows a door).

Fitted per entity (see include/campx_b200.h `cx_entity_desc`)
  kind (a drape that only ever loses the cell its watched entity stands on is a pickup; one that clears all of itself
  once a pickup drape is empty is a door), per-action toroidal move,
  blocker characters (one-cell drapes, and sprites that walls stop: PyColab's MazeWalker), per-action step reward,
  "entry" reward as a function of (action, character the last render showed at a watched entity's
  current cell), terminate directives per action or per (action, character under the watched entity)
  ("reach the goal"), default-discount directives per action, per-action visibility
  operation (sprites), per-action `change_z_order` calls; per game: the backdrop's per-action roll.
"""
import collections

import numpy as np
import torch

from .. import _native as N
from .. import things
from ..description import EntitySpec, GameSpec

ACTION_FORMATS = ("onehot_float", "onehot_list", "index")


class CompileError(NotImplementedError):
    """The game uses behaviour outside the kernel primitives."""


def encode_action(fmt, index, n_actions):
    """Discrete action index -> the object the world's update() methods expect."""
    if fmt == "index":
        return int(index)
    onehot = [0] * n_actions
    onehot[int(index)] = 1
    if fmt == "onehot_float":
        return torch.FloatTensor(onehot)           # boat_race.py:26,40 `actions.byte()`
    if fmt == "onehot_list":
        return onehot                              # Demo 1-3 `game.play([1,0,0,0,0])`
    raise ValueError("unknown action format %r" % (fmt,))


def _f32(x):
    if torch.is_tensor(x):
        x = x.item()
    return np.float32(x)


def _snapshot(shadow):
    snap = {}
    for ch, ent in shadow.things.items():
        if isinstance(ent, things.Sprite):
            snap[ch] = ("sprite", (int(ent.position[0]), int(ent.position[1])), bool(ent.visible))
        else:
            snap[ch] = ("drape", ent.curtain.as_subclass(torch.Tensor).detach().to(torch.int64).numpy().copy())
    return snap


class _Probe(object):
    __slots__ = ("action", "teleports", "pre", "post", "group_board", "after", "events", "reward", "discount",
                 "game_over", "backdrop_pre", "backdrop_post", "z_post", "hidden")


# attributes that ARE the modelled state of an entity (things.py:25-26,44-45,66-69) or compile-time plumbing
_MODELLED = frozenset(("_curtain", "_palette", "_character", "_corner", "_position", "_visible", "update"))


def _freeze(value):
    """A comparable rendering of an attribute value; None for values that cannot be compared reliably."""
    if torch.is_tensor(value):
        t = value.as_subclass(torch.Tensor).detach()
        return ("tensor", tuple(t.shape), str(t.dtype), t.cpu().numpy().tobytes())
    if isinstance(value, np.ndarray):
        return ("array", value.shape, str(value.dtype), value.tobytes())
    if isinstance(value, (bool, int, float, complex, str, bytes, type(None), np.generic)):
        return ("scalar", type(value).__name__, value if value == value else "nan")
    if isinstance(value, (list, tuple)):
        parts = tuple(_freeze(v) for v in value)
        return None if any(x is None for x in parts) else (type(value).__name__, parts)
    if isinstance(value, (set, frozenset)):
        parts = [_freeze(v) for v in value]
        return None if any(x is None for x in parts) else ("set", tuple(sorted(map(repr, parts))))
    if isinstance(value, dict):
        parts = {repr(k): _freeze(v) for k, v in value.items()}
        return None if any(x is None for x in parts.values()) else ("dict", tuple(sorted(parts.items())))
    return None


def _hidden_state(shadow):
    """Everything an entity (or the Plot) remembers besides the state the primitives model: instance attributes
    other than curtain / position / visibility, and non-tensor Plot entries (tensor entries are the usual aliases of
    renderer layers, examples/boat_race.py:59,91 -- functions of the last render, which IS modelled)."""
    out = {}
    ents = list(shadow.things.items()) + [("<backdrop>", shadow.backdrop)]
    for ch, ent in ents:
        for name, value in vars(ent).items():
            if name not in _MODELLED:
                out[(ch, name)] = _freeze(value)
    for key, value in shadow.the_plot.items():
        if not torch.is_tensor(value):
            out[("<plot>", repr(key))] = _freeze(value)
    return out


BACKDROP = "__backdrop__"          # teleport key: pre-roll the backdrop curtain by (d_row, d_col)


def _teleport(shadow, base_masks, ch, where):
    if ch == BACKDROP:
        cur = shadow.backdrop.curtain
        rolled = np.roll(cur.as_subclass(torch.Tensor).numpy(), (where[0], where[1]), axis=(0, 1)).copy()
        cur.copy_(torch.from_numpy(rolled).to(cur.dtype))
        return
    ent = shadow.things[ch]
    rows, cols = shadow.rows, shadow.cols
    if isinstance(ent, things.Sprite):
        ent._position = ent.Position(int(where[0]), int(where[1]))
        if len(where) > 2:
            ent._visible = bool(where[2])
        return
    cur = ent.curtain
    if where[0] == "mask":                  # ("mask", uint8 [rows, cols]): a pickup drape with some items taken
        cur.copy_(torch.from_numpy(np.asarray(where[1], dtype=np.uint8)).to(cur.dtype))
    elif where[0] == "cell":
        cur.zero_()
        if where[1] is not None:
            cur[where[1] // cols, where[1] % cols] = 1
    else:                                   # ("roll", dr, dc)
        rolled = np.roll(base_masks[ch], (where[1], where[2]), axis=(0, 1))
        cur.copy_(torch.from_numpy(rolled.astype(np.uint8)).to(cur.dtype))


def run_probe(base, base_masks, fmt, n_actions, action, teleports):
    s = base.clone()
    for ch, where in teleports.items():
        _teleport(s, base_masks, ch, where)
    if teleports:
        s.render()                          # make board/layers (and Plot aliases of them) consistent
    p = _Probe()
    p.action, p.teleports = action, dict(teleports)
    p.pre = _snapshot(s)
    hidden_pre = _hidden_state(s)
    p.backdrop_pre = s.backdrop.curtain.as_subclass(torch.Tensor).numpy().copy()
    p.group_board, p.after = {}, {}

    # trace hooks: the board each update group saw, and the world right after each entity updated
    groups = s.update_groups
    hooked = []
    for gname, ents in groups:
        for i, ent in enumerate(ents):
            orig = ent.update

            def wrapped(actions, board, layers, backdrop, all_things, the_plot, _orig=orig, _ent=ent,
                        _g=gname, _first=(i == 0)):
                if _first:
                    p.group_board[_g] = board.as_subclass(torch.Tensor).numpy().copy()
                _orig(actions, board, layers, backdrop, all_things, the_plot)
                p.after[_ent.character] = _snapshot(s)

            ent.update = wrapped
            hooked.append(ent)
    try:
        p.reward, p.discount = s.play(encode_action(fmt, action, n_actions))
    finally:
        for ent in hooked:
            del ent.update
    p.game_over = s.game_over
    hidden_post = _hidden_state(s)
    p.hidden = sorted(k for k in set(hidden_pre) | set(hidden_post)
                      if hidden_pre.get(k, ("absent",)) != hidden_post.get(k, ("absent",)))
    p.events = collections.defaultdict(list)
    for who, kind, payload in s.the_plot.events:
        p.events[who].append((kind, payload))
    p.post = _snapshot(s)
    p.backdrop_post = s.backdrop.curtain.as_subclass(torch.Tensor).numpy().copy()
    p.z_post = list(s.things.keys())
    return p


def _cell_of(mask):
    idx = np.flatnonzero(mask.reshape(-1))
    if len(idx) == 0:
        return None
    if len(idx) > 1 or mask.reshape(-1)[idx[0]] != 1:
        raise CompileError("a one-cell drape grew to %d cells / non-binary values" % len(idx))
    return int(idx[0])


def _signed(d, size):
    d %= size
    return d - size if d > size // 2 else d


def _find_roll(before, after):
    rows, cols = before.shape
    cands = sorted(((dr, dc) for dr in range(rows) for dc in range(cols)),
                   key=lambda s: abs(_signed(s[0], rows)) + abs(_signed(s[1], cols)))
    for dr, dc in cands:
        if np.array_equal(np.roll(before, (dr, dc), axis=(0, 1)), after):
            return _signed(dr, rows), _signed(dc, cols)
    return None


def compile_game(shadow, n_actions=5, action_format=None, max_episode_steps=0, auto_reset=True,
                 track_returns=False, occlusion_in_layers=True, performance_regions=None):
    """Fingerprint `shadow` (a not-yet-started ShadowEngine) and return its GameSpec.

    Runs the shadow's its_showtime() first (campx/engine.py:487-544); the resulting state is the
    per-episode initial state the kernels reset to.
    """
    rows, cols, A = shadow.rows, shadow.cols, int(n_actions)
    cells = rows * cols
    if not 1 <= A <= N.CX_MAX_ACTIONS:
        raise CompileError("num_actions must be in 1..%d" % N.CX_MAX_ACTIONS)
    first_reward, first_discount = shadow.its_showtime()
    base = shadow
    chars = "".join(sorted(base.layers.keys()))
    z_chars = list(base.things.keys())
    order = [ent.character for _, ents in base.update_groups for ent in ents]
    if sorted(order) != sorted(z_chars):
        raise CompileError("every sprite/drape must belong to exactly one update group")
    rank = {ch: i for i, ch in enumerate(order)}
    group_of, group_name = {}, {}
    for gi, (gname, ents) in enumerate(base.update_groups):
        for ent in ents:
            group_of[ent.character] = gi
            group_name[ent.character] = gname
    base_snap = _snapshot(base)
    base_masks = {ch: v[1].astype(np.uint8) for ch, v in base_snap.items() if v[0] == "drape"}
    for ch, m in base_masks.items():
        if not np.isin(m, (0, 1)).all():
            raise CompileError("drape %r has a non-binary curtain" % ch)

    # ---- action format ---------------------------------------------------------------------------
    # A format is usable if every update() runs with it; among usable formats prefer the first under
    # which the outcome depends on the action (a python list compared with `actions == 4` raises
    # nothing but also never matches, so every action would look the same).
    formats = (action_format,) if action_format else ACTION_FORMATS
    usable, last_err = [], None
    for cand in formats:
        try:
            trial = [run_probe(base, base_masks, cand, A, a, {}) for a in range(A)]
        except (CompileError, NotImplementedError):
            raise
        except Exception as e:  # the world's update() does not take this kind of action object
            last_err = e
            continue

        def outcome(pr):
            state = tuple((ch, v[1:] if v[0] == "sprite" else v[1].tobytes()) for ch, v in sorted(pr.post.items()))
            state += (pr.backdrop_post.tobytes(),)
            events = tuple((who, tuple((k, float(_f32(p)) if k == "reward" else p) for k, p in ev))
                           for who, ev in sorted(pr.events.items(), key=lambda kv: str(kv[0])))
            return state, events, pr.game_over

        usable.append((cand, trial, len(set(outcome(pr) for pr in trial)) > 1))
    if not usable:
        raise CompileError("no supported action format (%s) is accepted by this game's update() methods; "
                           "last error: %r" % (", ".join(formats), last_err))
    fmt, s0_probes, _ = next((u for u in usable if u[2]), usable[0])
    probes = list(s0_probes)

    def probe(action, teleports):
        pr = run_probe(base, base_masks, fmt, A, action, teleports)
        probes.append(pr)
        return pr

    # ---- classify entities -------------------------------------------------------------------------
    kind, moves = {}, {}
    for ch in z_chars:
        tag = base_snap[ch][0]
        if tag == "sprite":
            kind[ch] = N.CX_KIND_SPRITE
            continue
        m0 = base_masks[ch]
        changed = [not np.array_equal(pr.post[ch][1], m0) for pr in s0_probes]
        if not any(changed):
            kind[ch] = N.CX_KIND_STATIC
        elif all(_cleared_only(m0, pr.post[ch][1]) for pr in s0_probes):
            kind[ch] = N.CX_KIND_PICKUP          # only ever loses cells: collectible items (fitted below)
        elif int(m0.sum()) == 1:
            kind[ch] = N.CX_KIND_CELL
        else:
            kind[ch] = N.CX_KIND_ROLL

    # ---- sprites: per-action displacement, verified from corners; else a move + blocker fit ------------
    visible_ops, blockers = {}, {}
    for ch in [c for c in z_chars if kind[c] == N.CX_KIND_SPRITE]:
        p0, vis0 = base_snap[ch][1], base_snap[ch][2]
        mv = []
        for pr in s0_probes:
            q = pr.post[ch][1]
            mv.append((_signed(q[0] - p0[0], rows), _signed(q[1] - p0[1], cols)))
        moves[ch] = mv
        # Sprite._visible (things.py:320): per action keep / show / hide / toggle.  If it ever changes from the
        # initial state, every action is also probed from the other state (keep vs show are told apart there).
        seen = {a: {(vis0, s0_probes[a].post[ch][2])} for a in range(A)}
        if any(pr.post[ch][2] != vis0 for pr in s0_probes):
            for a in range(A):
                pr = probe(a, {ch: (p0[0], p0[1], not vis0)})
                seen[a].add((not vis0, pr.post[ch][2]))
        ops = []
        for a in range(A):
            fits = [op for op, fn in ((N.CX_VIS_KEEP, lambda v: v), (N.CX_VIS_SHOW, lambda v: True),
                                      (N.CX_VIS_HIDE, lambda v: False), (N.CX_VIS_TOGGLE, lambda v: not v))
                    if all(fn(pre) == post for pre, post in seen[a])]
            if not fits:
                raise CompileError("sprite %r: action %d changes its visibility in a way that is not "
                                   "keep/show/hide/toggle" % (ch, a))
            ops.append(fits[0])
        visible_ops[ch] = ops
        model_vis = lambda a, v, _ops=ops: {N.CX_VIS_KEEP: v, N.CX_VIS_SHOW: True, N.CX_VIS_HIDE: False,
                                            N.CX_VIS_TOGGLE: not v}[_ops[a]]
        spots = {(0, 0), (rows - 1, cols - 1), (0, cols - 1), (rows - 1, 0), (rows // 2, cols // 2)}
        miss = None
        for spot in sorted(spots):
            for a in range(A):
                pr = probe(a, {ch: spot})
                want = ((spot[0] + mv[a][0]) % rows, (spot[1] + mv[a][1]) % cols)
                if pr.post[ch][1] != want and miss is None:
                    miss = "from %s action %d: got %s, model %s" % (spot, a, pr.post[ch][1], want)
                if pr.post[ch][2] != model_vis(a, pr.pre[ch][2]):
                    raise CompileError("sprite %r: its visibility depends on more than the action" % ch)
        if miss is not None:       # not a fixed displacement: a sprite that walls stop (PyColab's MazeWalker)?
            moves[ch], blockers[ch] = _fit_blocked_sprite(ch, miss, p0, ops, probes, s0_probes, probe, group_name[ch],
                                                          A, rows, cols)

    # ---- rolling drapes -----------------------------------------------------------------------------
    for ch in [c for c in z_chars if kind[c] == N.CX_KIND_ROLL]:
        m0 = base_masks[ch]
        mv = []
        for pr in s0_probes:
            sh = _find_roll(m0, pr.post[ch][1].astype(np.uint8))
            if sh is None:
                raise CompileError("drape %r changes its mask in a way that is neither static, a one-cell "
                                   "move nor a toroidal roll" % ch)
            mv.append(sh)
        moves[ch] = mv
        for off in sorted({(rows - 1, cols - 1), (1, 0), (0, 1), (rows // 2, cols // 3)}):
            for a in range(A):
                pr = probe(a, {ch: ("roll", off[0], off[1])})
                want = np.roll(m0, (off[0] + mv[a][0], off[1] + mv[a][1]), axis=(0, 1))
                if not np.array_equal(pr.post[ch][1].astype(np.uint8), want):
                    raise CompileError("drape %r does not roll by a fixed shift per action" % ch)

    # ---- one-cell drapes: BFS over reachable cells, move + blocker fit ---------------------------------
    reached, observed = {}, {}                     # per one-cell drape: cells reached, [(p, a, q, probe)]
    for ch in [c for c in z_chars if kind[c] == N.CX_KIND_CELL]:
        p0 = _cell_of(base_masks[ch])
        seen, queue, trans = {p0}, collections.deque([p0]), []
        while queue:
            p = queue.popleft()
            for a in range(A):
                pr = s0_probes[a] if p == p0 else probe(a, {ch: ("cell", p)})
                q = _cell_of(pr.post[ch][1])
                trans.append((p, a, q, pr))
                if q is not None and q not in seen:
                    if len(seen) >= N.CX_MAX_CELLS:
                        raise CompileError("reachable set too large")
                    seen.add(q)
                    queue.append(q)
        moves[ch], blockers[ch] = _fit_cell_drape(ch, trans, group_name[ch], A, rows, cols)
        reached[ch], observed[ch] = seen, trans

    # ---- pickup drapes: items the agent collects; door drapes: opened once a pickup drape is empty ----------
    # A drape that looked static from the initial state may still lose an item once the agent stands elsewhere.
    for ch in z_chars:
        if kind[ch] == N.CX_KIND_STATIC and any(
                not np.array_equal(pr.post[ch][1], pr.pre[ch][1]) for pr in probes) and all(
                _cleared_only(pr.pre[ch][1], pr.post[ch][1]) for pr in probes):
            kind[ch] = N.CX_KIND_PICKUP
    pickups, doors = {}, {}
    if any(k == N.CX_KIND_PICKUP for k in kind.values()):
        agent = _pickup_agent(z_chars, kind, rows, cols, len(base.update_groups), performance_regions,
                              occlusion_in_layers)
        probed = []
        while True:
            # a drape that only ever loses the cell the agent stands on is a pickup; one that changes otherwise (a
            # whole door opening) may be a door.  The probes with pickup drapes emptied show more of both: a pickup
            # behind a door, a door that updates before its key.
            for ch in z_chars:
                if kind[ch] in (N.CX_KIND_STATIC, N.CX_KIND_PICKUP) and any(
                        not np.array_equal(pr.post[ch][1], pr.pre[ch][1]) for pr in probes):
                    kind[ch] = N.CX_KIND_PICKUP if all(
                        _cleared_only(pr.pre[ch][1], pr.post[ch][1]) and _takes_the_agents_cell(pr, ch, agent)
                        for pr in probes) else N.CX_KIND_DOOR
            keys = [c for c in z_chars if kind[c] == N.CX_KIND_PICKUP]
            fresh = [k for k in keys if k not in probed]
            if not fresh:
                break
            _check_pickup_cells(z_chars, kind, agent, base_masks)
            scenes = [(k,) for k in fresh] + ([tuple(keys)] if len(keys) > 1 else [])
            _probe_emptied(scenes, fresh, agent, z_chars, kind, base_masks, reached, observed, probe, A, rows, cols)
            probed += fresh
        pickups = _fit_pickups(z_chars, kind, agent, base_masks, probes, probe, A, rows, cols)
        doors = _fit_doors(z_chars, kind, agent, keys, base_masks, probes, rank)
        # the agent's move and blockers, checked (and its blockers completed) behind the opened doors too
        moves[agent], blockers[agent] = _fit_cell_drape(agent, observed[agent], group_name[agent], A, rows, cols)

    # ---- backdrop: static apart from the sprite stamps of quirk Q1, or rolled by Backdrop.update() ------------
    def first_drape_of(order_):
        return next((i for i, c in enumerate(order_) if kind[c] != N.CX_KIND_SPRITE), len(order_))

    any_drape = first_drape_of(z_chars) < len(z_chars)
    backdrop_moves = None
    s0_changed = [not np.array_equal(pr.backdrop_pre, pr.backdrop_post) for pr in s0_probes]
    stamp_cells_only = True
    for pr in s0_probes:
        for r, c in np.argwhere(pr.backdrop_pre != pr.backdrop_post):
            if not any(kind[s_] == N.CX_KIND_SPRITE and pr.post[s_][1] == (int(r), int(c)) and
                       pr.backdrop_post[r, c] == ord(s_) for s_ in z_chars):
                stamp_cells_only = False
    if any(s0_changed) and any_drape and not stamp_cells_only:
        # things.py:103-148 Backdrop.update(): fitted as a per-action toroidal roll of the curtain (scrolling scenery)
        bd0 = s0_probes[0].backdrop_pre
        backdrop_moves = []
        for pr in s0_probes:
            sh = _find_roll(bd0, pr.backdrop_post)
            if sh is None:
                raise CompileError("Backdrop.update() changes the backdrop in a way that is not a toroidal roll "
                                   "of its curtain")
            backdrop_moves.append(sh)
        for off in sorted({(rows - 1, cols - 1), (1, 0), (0, 1), (rows // 2, cols // 3)}):
            for a in range(A):
                pr = probe(a, {BACKDROP: off})
                want = np.roll(pr.backdrop_pre, backdrop_moves[a], axis=(0, 1))
                if not np.array_equal(pr.backdrop_post, want):
                    raise CompileError("Backdrop.update() does not roll the backdrop by a fixed shift per action")
    for pr in probes:
        if pr.events.get(None):
            raise CompileError("Backdrop.update() issues plot directives (%s); not supported"
                               % ", ".join(sorted({k for k, _ in pr.events[None]})))
        if backdrop_moves is not None:
            if BACKDROP not in pr.teleports and not np.array_equal(
                    pr.backdrop_post, np.roll(pr.backdrop_pre, backdrop_moves[pr.action], axis=(0, 1))):
                raise CompileError("Backdrop.update() does not roll the backdrop by a fixed shift per action")
            continue
        # sprites that lie, visibly, behind the first drape of the initial or the resulting z-order stamp
        # their character into the backdrop (SURVEY quirk Q1)
        allowed = set()
        for order_ in (z_chars, pr.z_post):
            fd = first_drape_of(order_)
            if fd < len(order_):
                allowed.update(c for c in order_[:fd] if pr.post[c][2])
        for r, c in np.argwhere(pr.backdrop_pre != pr.backdrop_post):
            ok = any(pr.post[s_][1] == (int(r), int(c)) and pr.backdrop_post[r, c] == ord(s_) for s_ in allowed)
            if not ok and any_drape:
                raise CompileError("Backdrop.update() changes the backdrop in a way that is neither a sprite stamp "
                                   "nor a roll of the whole curtain")

    # ---- hidden state: behaviour the primitives cannot see --------------------------------------------------------
    # Every probe starts from a copy of the its_showtime state, so an entity that counts steps, remembers visits or
    # draws random numbers would look stateless here and compile to something that diverges later.  Any instance
    # attribute (other than curtain / position / visibility) or non-tensor Plot entry that a step changes is such
    # state: refuse the game instead of compiling it wrongly.
    for pr in probes:
        if pr.hidden:
            owner, name = pr.hidden[0]
            raise CompileError("%s keeps state the kernel primitives do not model: %s changed during a step (action "
                               "%d).  Entities may only depend on curtains, positions, visibility, the last render "
                               "and the action." % ("the Plot" if owner == "<plot>" else
                                                    "the Backdrop" if owner == "<backdrop>" else "entity %r" % owner,
                                                    name if owner == "<plot>" else "attribute %r" % name, pr.action))

    # ---- rewards, terminate, discount ----------------------------------------------------------------------
    movers = [c for c in z_chars if kind[c] in (N.CX_KIND_CELL, N.CX_KIND_SPRITE)]

    def seen_under(pr, ch, w):
        """Character the last render (the one entity `ch`'s update group saw) showed at mover `w`'s cell as of right
        after `ch` updated (things[w] is current sibling state, boat_race.py:79); None for an empty mask."""
        snap = pr.after[ch][w]
        cell = snap[1][0] * cols + snap[1][1] if snap[0] == "sprite" else _cell_of(snap[1])
        return None if cell is None else chr(int(pr.group_board[group_name[ch]].reshape(-1)[cell]))

    specs = []
    for z, ch in enumerate(z_chars):
        if ch in pickups:
            agent, reward, emptied = pickups[ch]
            specs.append(EntitySpec(character=ch, kind=N.CX_KIND_PICKUP, mask=base_masks[ch], update_rank=rank[ch],
                                    update_group=group_of[ch], watch=agent,
                                    entry_reward={a: {ch: reward[a]} for a in range(A)}, terminate_emptied=emptied))
            continue
        if ch in doors:
            specs.append(EntitySpec(character=ch, kind=N.CX_KIND_DOOR, mask=base_masks[ch], update_rank=rank[ch],
                                    update_group=group_of[ch], door_key=doors[ch]))
            continue
        obs = []                                  # (probe, action, f32 reward or None)
        term, disc, zord = {}, {}, {}
        for pr in probes:
            val = None
            zs = []
            for k, payload in pr.events.get(ch, ()):
                if k == "reward":
                    val = _f32(payload) if val is None else np.float32(_f32(payload) + val)
                elif k == "z_order":
                    zs.append(tuple(payload))
            zord.setdefault(pr.action, set()).add(tuple(zs))
            obs.append((pr, pr.action, val))
            t = [payload for k, payload in pr.events.get(ch, ()) if k == "terminate"]
            d = [payload for k, payload in pr.events.get(ch, ()) if k == "discount"]
            term.setdefault(pr.action, set()).add(t[-1] if t else None)
            disc.setdefault(pr.action, set()).add(d[-1] if d else None)
        for a, vals in disc.items():
            if len(vals) != 1:
                raise CompileError("entity %r calls change_default_discount for action %d only in some states" % (ch, a))
        # terminate_episode: per action, or -- "reach the goal" games -- per (action, character the last render
        # showed under a moving entity), the same query entry rewards use
        term_watch, terminate_on = None, {}
        if any(len(vals) != 1 for vals in term.values()):
            for w in movers:
                table, ok = {}, True
                for pr in probes:
                    t = [payload for k, payload in pr.events.get(ch, ()) if k == "terminate"]
                    table.setdefault((pr.action, seen_under(pr, ch, w)), set()).add(t[-1] if t else None)
                if all(len(v) == 1 for v in table.values()):
                    term_watch = w
                    for (a, seen_char), v in table.items():
                        value = next(iter(v))
                        if value is not None:
                            if seen_char is None:
                                raise CompileError("entity %r terminates the episode while %r has an empty mask" % (ch, w))
                            terminate_on.setdefault(a, {})[seen_char] = float(value)
                    break
            if term_watch is None:
                raise CompileError("entity %r calls terminate_episode depending on something other than (action, "
                                   "what the last render showed under a moving entity)" % ch)
            for a in list(terminate_on):       # fires for every character seen => unconditional for that action
                seen_all = {k for (aa, k) in table if aa == a}
                if set(terminate_on[a]) == seen_all and len(set(terminate_on[a].values())) == 1 and len(term[a]) == 1:
                    del terminate_on[a]
            for a in terminate_on:
                term[a] = {None}               # not an unconditional directive of this action
        z_orders = {}
        for a, vals in zord.items():
            if len(vals) != 1:
                raise CompileError("entity %r calls change_z_order for action %d only in some states" % (ch, a))
            calls = list(next(iter(vals)))
            for move_this, front_of in calls:
                for c in (move_this,) if front_of is None else (move_this, front_of):
                    if c not in z_chars:       # engine.py:247-262
                        raise CompileError("A z-order change directive names character %r, but no such Sprite or "
                                           "Drape exists" % (c,))
                if move_this == front_of:
                    raise CompileError("change_z_order(%r, %r) would drop the entity from the game "
                                       "(engine.py:270-279); not supported" % (move_this, front_of))
            if calls:
                z_orders[a] = calls
        terminate = {a: next(iter(v)) for a, v in term.items() if len(v) == 1 and next(iter(v)) is not None}
        for a in terminate_on:
            if a in disc and next(iter(disc[a])) is not None:
                raise CompileError("entity %r both changes the default discount and conditionally terminates the "
                                   "episode for action %d" % (ch, a))
        discount = {a: next(iter(v)) for a, v in disc.items() if next(iter(v)) is not None and a not in terminate}

        step_reward, watch, entry = None, None, None
        has = {}
        for pr, a, val in obs:
            has.setdefault(a, set()).add(val is not None)
        for a, hv in has.items():
            if len(hv) != 1:
                raise CompileError("entity %r calls add_reward for action %d only in some states" % (ch, a))
        if any(next(iter(hv)) for hv in has.values()):
            by_action = {}
            for pr, a, val in obs:
                if val is not None:
                    by_action.setdefault(a, set()).add(float(val))
            if all(len(v) == 1 for v in by_action.values()):
                step_reward = [next(iter(by_action[a])) if a in by_action else None for a in range(A)]
            else:
                fitted = None
                for w in ([term_watch] if term_watch is not None else movers):   # one `watch` per entity
                    table, ok = {}, True
                    for pr, a, val in obs:
                        if val is None:
                            continue
                        table.setdefault((a, seen_under(pr, ch, w)), set()).add(float(val))
                    if all(len(v) == 1 for v in table.values()):
                        fitted = (w, {k: next(iter(v)) for k, v in table.items()})
                        break
                if fitted is None:
                    raise CompileError("the reward of entity %r depends on something other than (action, what the "
                                       "last render showed under a moving entity)" % ch)
                watch, table = fitted
                step_reward, entry = [], {}
                for a in range(A):
                    vals = {k: v for (aa, k), v in table.items() if aa == a}
                    if not vals:
                        step_reward.append(None)
                        continue
                    if watch in vals:            # the watched entity seen in place: nothing was entered
                        basev = vals[watch]
                    elif None in vals:
                        basev = vals[None]
                    else:
                        basev = collections.Counter(vals.values()).most_common(1)[0][0]
                    step_reward.append(basev)
                    for k, v in vals.items():
                        if k is None:
                            if v != basev:
                                raise CompileError("entity %r pays a different reward when %r has an empty mask"
                                                   % (ch, watch))
                            continue
                        if v != basev:
                            extra = float(np.float32(v) - np.float32(basev))
                            if np.float32(np.float32(basev) + np.float32(extra)) != np.float32(v):
                                raise CompileError("reward of %r is not exactly representable as base+entry" % ch)
                            entry.setdefault(a, {})[k] = extra
        snap = base_snap[ch]
        specs.append(EntitySpec(
            character=ch, kind=kind[ch],
            mask=(base_masks[ch] if snap[0] == "drape" else np.zeros((rows, cols), np.uint8)),
            update_rank=rank[ch], update_group=group_of[ch],
            visible=(snap[2] if snap[0] == "sprite" else True),
            init_pos=(snap[1] if snap[0] == "sprite" else None),
            moves=moves.get(ch), blockers=blockers.get(ch, ""),
            step_reward=step_reward, watch=watch if watch is not None else term_watch, entry_reward=entry,
            terminate=terminate or None, terminate_on=terminate_on or None, discount=discount or None,
            visible_op=visible_ops.get(ch), z_orders=z_orders or None))

    if pickups:
        _check_pickup_game(specs, pickups, base.backdrop.curtain.as_subclass(torch.Tensor).numpy(), backdrop_moves,
                           rows, cols)

    # ---- whole-step consistency: the per-entity fits must add up to what play() returned --------------------
    spec = GameSpec(rows=rows, cols=cols, chars=chars, n_actions=A, entities=specs,
                    backdrop=base.backdrop.curtain.as_subclass(torch.Tensor).numpy().astype(np.uint8).copy(),
                    n_groups=len(base.update_groups), max_episode_steps=max_episode_steps,
                    auto_reset=auto_reset, track_returns=track_returns,
                    first_reward=None if first_reward is None else float(_f32(first_reward)),
                    first_discount=float(first_discount), action_format=fmt, backdrop_moves=backdrop_moves,
                    occlusion_in_layers=bool(occlusion_in_layers), performance_regions=performance_regions)
    spec.n_probes = len(probes)
    return spec


def _fit_blocked_sprite(ch, miss, p0, ops, probes, s0_probes, probe, group, A, rows, cols):
    """A sprite that is no fixed toroidal displacement per action (`miss` says where that model failed), fitted as a
    blocked sprite: action a targets position + moves[a] (toroidal) and stays put where the last render (the board of
    the sprite's update group) showed one of the blocker characters there.  Breadth-first search over the positions
    reachable from `p0`, then the model is checked on every probe so far.  Returns (moves, blockers)."""
    if any(op != N.CX_VIS_KEEP for op in ops):
        raise CompileError("sprite %r does not move by a fixed toroidal displacement per action (%s), and a sprite "
                           "that walls stop must keep its visibility" % (ch, miss))
    seen, queue, trans = {p0}, collections.deque([p0]), {}
    while queue:
        p = queue.popleft()
        for a in range(A):
            pr = s0_probes[a] if p == p0 else probe(a, {ch: p})
            q = pr.post[ch][1]
            trans[(p, a)] = q
            if q not in seen:
                seen.add(q)
                queue.append(q)
    mv = []
    for a in range(A):
        deltas = {(_signed(q[0] - p[0], rows), _signed(q[1] - p[1], cols))
                  for (p, aa), q in trans.items() if aa == a and q != p}
        if len(deltas) > 1:
            raise CompileError("sprite %r: action %d moves it by different amounts %s" % (ch, a, sorted(deltas)))
        mv.append(deltas.pop() if deltas else (0, 0))

    def target(p, a):
        return ((p[0] + mv[a][0]) % rows, (p[1] + mv[a][1]) % cols)

    blk = set()
    for pr in probes:
        p, q = pr.pre[ch][1], pr.post[ch][1]
        t = target(p, pr.action)
        if t != p and q != t:
            blk.add(chr(int(pr.group_board[group][t])))
    for pr in probes:                            # the fitted model must reproduce every observation
        p, q = pr.pre[ch][1], pr.post[ch][1]
        t = target(p, pr.action)
        model = p if chr(int(pr.group_board[group][t])) in blk else t
        if model != q:
            raise CompileError("sprite %r does not move by a fixed toroidal displacement per action (%s), nor as a "
                               "sprite that walls stop: from %s action %d the model (move %s, blockers %r) predicts %s "
                               "but update() gave %s" % (ch, miss, p, pr.action, mv[pr.action], "".join(sorted(blk)),
                                                         model, q))
    return mv, "".join(sorted(blk))


def _cleared_only(before, after):
    """`after` is `before` with zero or more cells cleared (a binary curtain that only loses cells)."""
    before, after = np.asarray(before).reshape(-1), np.asarray(after).reshape(-1)
    return bool(np.isin(after, (0, 1)).all() and np.all(after <= (before != 0)))


def _pickup_agent(z_chars, kind, rows, cols, n_groups, performance_regions, occlusion_in_layers):
    """The one-cell drape agent of a game with CX_KIND_PICKUP candidates; refuses any other kind of game."""
    chars = [c for c in z_chars if kind[c] == N.CX_KIND_PICKUP]
    cells_ = [c for c in z_chars if kind[c] == N.CX_KIND_CELL]
    for ch in chars:
        if len(cells_) != 1 or any(kind[c] in (N.CX_KIND_SPRITE, N.CX_KIND_ROLL) for c in z_chars) or n_groups > 1 \
                or rows * cols > 254:
            raise CompileError("pickup drape %r needs a single-agent game (one moving one-cell drape over a static "
                               "scene, one update group, at most 254 cells); this game would run on the generic "
                               "kernels" % ch)
        if performance_regions is not None:
            raise CompileError("pickup drape %r together with performance_regions is not supported" % ch)
        if not occlusion_in_layers:
            raise CompileError("pickup drape %r needs occluded layers (occlusion_in_layers=True)" % ch)
    return cells_[0]


def _check_pickup_cells(z_chars, kind, agent, base_masks):
    """Where the items of the CX_KIND_PICKUP drapes may lie: below the agent, one drape per cell, none under the agent's
    initial cell, at most CX_MAX_PICKUPS in all."""
    z = {c: i for i, c in enumerate(z_chars)}
    agent_cell = _cell_of(base_masks[agent])
    owner, total = {}, 0
    for ch in [c for c in z_chars if kind[c] == N.CX_KIND_PICKUP]:
        if z[ch] > z[agent]:
            raise CompileError("pickup drape %r lies in front of the agent %r in z-order; it must be below it"
                               % (ch, agent))
        for c in np.flatnonzero(base_masks[ch].reshape(-1)):
            if c in owner:
                raise CompileError("pickup drapes %r and %r share cell %d" % (owner[c], ch, c))
            if c == agent_cell:
                raise CompileError("pickup drape %r has an item under the agent's initial cell" % ch)
            owner[c] = ch
            total += 1
        if total > N.CX_MAX_PICKUPS:
            raise CompileError("more than %d item cells in all (pickup drape %r)" % (N.CX_MAX_PICKUPS, ch))


def _fit_cell_drape(ch, trans, group, A, rows, cols):
    """Per-action move and blocker characters of one-cell drape `ch` from its observed transitions [(p, a, q, probe)]:
    action a moves it by one fixed toroidal delta, and a target cell that showed a blocker in the last render (the
    board of its update group) keeps it where it was drawn (nowhere when it was not drawn).  The model must reproduce
    every observation."""
    mv = []
    for a in range(A):
        deltas = set()
        for p, aa, q, _ in trans:
            if aa == a and q is not None and q != p:
                deltas.add((_signed(q // cols - p // cols, rows), _signed(q % cols - p % cols, cols)))
        if len(deltas) > 1:
            raise CompileError("drape %r: action %d moves it by different amounts %s" % (ch, a, sorted(deltas)))
        mv.append(deltas.pop() if deltas else (0, 0))
    blk = set()

    def target(p, a):
        return ((p // cols + mv[a][0]) % rows) * cols + (p % cols + mv[a][1]) % cols

    for p, a, q, pr in trans:
        t = target(p, a)
        if t != p and q != t:
            seen_char = int(pr.group_board[group].reshape(-1)[t])
            blk.add(chr(seen_char))
    for p, a, q, pr in trans:     # the fitted model must reproduce every observation
        board = pr.group_board[group].reshape(-1)
        t = target(p, a)
        vis = int(board[p]) == ord(ch)
        blocked = chr(int(board[t])) in blk
        model = (p if vis else None) if blocked else t
        if model != q:
            raise CompileError("drape %r: from cell %d action %d the model (move %s, blockers %r) predicts "
                               "%s but update() gave %s" % (ch, p, a, mv[a], "".join(sorted(blk)), model, q))
    return mv, "".join(sorted(blk))


def _takes_the_agents_cell(pr, ch, agent):
    """In probe `pr`, drape `ch` lost at most the cell the agent stood on as `ch` updated (the pickup rule)."""
    pre, post = pr.pre[ch][1].reshape(-1), pr.post[ch][1].reshape(-1)
    c = _cell_of(pr.after[ch][agent][1])
    model = pre.copy()
    if c is not None:
        model[c] = 0
    return np.array_equal(post, pre) or np.array_equal(post, model)


def _probe_emptied(scenes, keys, agent, z_chars, kind, base_masks, reached, observed, probe, A, rows, cols):
    """Probes of the states the initial one does not show: the pickup drapes of each scene emptied, with whatever that
    opened open, every action from every cell the agent reaches there by breadth-first search (starting from every
    cell it reached before); and each of `keys` holding one item only, every action from the agent's start.  Every fit
    runs on them: a door opens in them, the cells behind it are reached, and an entity that depends on a drape's
    emptying some other way is refused.  The agent's transitions go to `observed`, the cells it reached to
    `reached`."""
    cells = reached[agent]
    for emptied in scenes:
        scene = {k: ("mask", np.zeros((rows, cols), np.uint8)) for k in emptied}
        seed = probe(A - 1, dict(scene))          # one step on: the drapes that open when these are empty are open
        for c in z_chars:
            if kind[c] in (N.CX_KIND_STATIC, N.CX_KIND_DOOR) and not np.array_equal(seed.post[c][1], seed.pre[c][1]):
                scene[c] = ("mask", seed.post[c][1].astype(np.uint8))
        seen, queue = set(cells), collections.deque(sorted(cells))
        while queue:
            p = queue.popleft()
            for a in range(A):
                pr = probe(a, dict(scene, **{agent: ("cell", p)}))
                q = _cell_of(pr.post[agent][1])
                observed[agent].append((p, a, q, pr))
                if q is not None and q not in seen:
                    seen.add(q)
                    queue.append(q)
        cells |= seen
    for k in keys:
        for c in np.flatnonzero(base_masks[k].reshape(-1)):
            one = np.zeros(rows * cols, np.uint8)
            one[c] = 1
            for a in range(A):
                probe(a, {k: ("mask", one.reshape(rows, cols))})


def _fit_doors(z_chars, kind, agent, keys, base_masks, probes, rank):
    """Fit every CX_KIND_DOOR candidate D: a drape whose curtain stays what it was while one pickup drape K (its key)
    still holds an item as D updates, and is empty from the first update that finds K empty on; D calls no plot
    directive.  Returns {door char: key char}."""
    z = {c: i for i, c in enumerate(z_chars)}
    out = {}
    for ch in [c for c in z_chars if kind[c] == N.CX_KIND_DOOR]:
        def opens_with(k):
            for pr in probes:
                pre, post = pr.pre[ch][1], pr.post[ch][1]
                if not np.array_equal(post, pre if pr.after[ch][k][1].any() else np.zeros_like(pre)):
                    return False
            return True
        key = next((k for k in keys if opens_with(k)), None)
        if key is None:
            raise CompileError("drape %r changes its curtain in a way that is neither static, a pickup nor a door (a "
                               "door keeps its whole curtain while one pickup drape holds an item, and clears all of it "
                               "once that drape is empty)" % ch)
        events = sorted({k for pr in probes for k, _ in pr.events.get(ch, ())})
        if events:
            raise CompileError("door drape %r calls %s; a door may call no plot directive" % (ch, events))
        if rank[ch] < rank[key]:
            raise CompileError("door drape %r updates before its key drape %r, so it opens one step after the key is "
                               "taken; a door must update after its key" % (ch, key))
        if z[ch] > z[agent]:
            raise CompileError("door drape %r lies in front of the agent %r in z-order; it must be below it"
                               % (ch, agent))
        m = base_masks[ch].reshape(-1) != 0
        for k in keys:
            if (m & (base_masks[k].reshape(-1) != 0)).any():
                raise CompileError("door drape %r shares a cell with an item of pickup drape %r" % (ch, k))
        if m[_cell_of(base_masks[agent])]:
            raise CompileError("door drape %r covers the agent's initial cell" % ch)
        for other in out:
            if (m & (base_masks[other].reshape(-1) != 0)).any():
                raise CompileError("door drapes %r and %r share a cell" % (other, ch))
        out[ch] = key
        if len(out) > N.CX_MAX_DOORS:
            raise CompileError("more than %d door drapes (door drape %r)" % (N.CX_MAX_DOORS, ch))
    return out


def _fit_pickups(z_chars, kind, agent, base_masks, probes, probe, A, rows, cols):
    """Fit every CX_KIND_PICKUP candidate: when its update() runs and its curtain holds the watched agent's current
    cell (the entry-reward query: the post-move cell if it updates after the agent, the pre-move cell otherwise), it
    clears that one cell and calls add_reward(r[a]); if that emptied the curtain it may call terminate_episode(v);
    nothing else.  Probes are added with the item already taken and with it as the last one.  Returns
    {char: (agent char, [r[a]], v or None)}."""
    chars = [c for c in z_chars if kind[c] == N.CX_KIND_PICKUP]

    def watched(pr, ch):
        return _cell_of(pr.after[ch][agent][1])

    out = {}
    for ch in chars:
        m0 = base_masks[ch].reshape(-1)
        for pr in [pr for pr in probes if ch not in pr.teleports]:
            c = watched(pr, ch)
            if c is None or not m0[c]:
                continue
            taken, last = m0.copy(), np.zeros_like(m0)
            taken[c], last[c] = 0, 1
            for m in (taken, last):
                probe(pr.action, dict(pr.teleports, **{ch: ("mask", m.reshape(rows, cols))}))
        rewards, emptied = {}, set()
        for pr in probes:
            pre, post = pr.pre[ch][1].reshape(-1), pr.post[ch][1].reshape(-1)
            c = watched(pr, ch)
            hit = c is not None and pre[c] != 0
            model = pre.copy()
            if hit:
                model[c] = 0
            if not np.array_equal(post, model):
                raise CompileError("drape %r changes its curtain in a way that is neither static nor a pickup "
                                   "(clearing the cell %r stands on)" % (ch, agent))
            events = pr.events.get(ch, ())
            if not hit:
                if events:
                    raise CompileError("pickup drape %r calls %s in a step that takes no item"
                                       % (ch, sorted({k for k, _ in events})))
                continue
            paid = [p for k, p in events if k == "reward"]
            ends = [p for k, p in events if k == "terminate"]
            if len(paid) != 1 or len(paid) + len(ends) != len(events):
                raise CompileError("pickup drape %r must call add_reward exactly once when it takes an item, and "
                                   "nothing but terminate_episode besides" % ch)
            rewards.setdefault(pr.action, set()).add(float(_f32(paid[0])))
            if model.any():
                if ends:
                    raise CompileError("pickup drape %r calls terminate_episode while items remain" % ch)
            else:
                emptied.add(float(ends[-1]) if ends else None)
        values = set().union(*rewards.values())
        if any(len(v) != 1 for v in rewards.values()) or (len(rewards) < A and len(values) != 1):
            raise CompileError("the reward of pickup drape %r depends on something other than the action" % ch)
        if len(emptied) != 1:
            raise CompileError("pickup drape %r calls terminate_episode only sometimes when it takes its last item" % ch)
        reward = [next(iter(rewards.get(a, values))) for a in range(A)]
        out[ch] = (agent, reward, emptied.pop())
    return out


def _check_pickup_game(specs, pickups, backdrop, backdrop_moves, rows, cols):
    """Refuse pickup games the single-agent kernels cannot run exactly: a changing render state, or another entity
    that depends on whether an item is present (an item, or what lies under it, among its blockers, entry-reward or
    terminate characters)."""
    for e in specs:
        if e.z_orders or (backdrop_moves and any(m != (0, 0) for m in backdrop_moves)):
            raise CompileError("pickup drape %r needs a static render order and backdrop (%r changes it)"
                               % (next(iter(pickups)), e.character))
    present, absent = backdrop.reshape(-1).astype(np.int64), backdrop.reshape(-1).astype(np.int64)
    for e in specs:
        if e.kind in (N.CX_KIND_STATIC, N.CX_KIND_PICKUP):
            m = np.asarray(e.mask).reshape(-1) != 0
            present = np.where(m, ord(e.character), present)
            if e.kind == N.CX_KIND_STATIC:
                absent = np.where(m, ord(e.character), absent)
    items = {}
    for e in specs:
        if e.kind == N.CX_KIND_PICKUP:
            for c in np.flatnonzero(np.asarray(e.mask).reshape(-1)):
                if present[c] != absent[c]:
                    items.setdefault(e.character, set()).update((chr(present[c]), chr(absent[c])))
    for e in specs:
        if e.kind == N.CX_KIND_PICKUP:
            continue
        seen = set(e.blockers)
        for table in list((e.entry_reward or {}).values()) + list((e.terminate_on or {}).values()):
            seen.update(table)
        for ch, shown in items.items():
            if seen & shown:
                raise CompileError("entity %r depends on whether an item of pickup drape %r is present (%r among its "
                                   "blockers, entry-reward or terminate characters)"
                                   % (e.character, ch, "".join(sorted(seen & shown))))
