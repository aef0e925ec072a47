"""The batched game engine: CampX's `Engine` API over hand-written CUDA kernels.

Public surface mirrors `campx/engine.py`: set-up methods `update_group` (:352-365), `add_sprite`
(:43-66), `add_prefilled_drape` (:367-404), `set_z_order` (:406-430), `set_prefilled_backdrop`
(:433-485) with the same validation and exception classes; `its_showtime()` (:487-544);
`play(actions)` (:114-166); `Palette` (:546-641).  `Engine.send/share` (PySyft, :68-112) are out of
scope.

New keyword arguments (everything else is the reference's):
    num_envs            number of independent environments stepped per `play()`; None = exactly one
                        environment with the reference's unbatched shapes and error behaviour
    device              CUDA device (default: current)
    num_actions         size of the discrete action set (default 5: left,right,up,down,stay,
                        examples/boat_race.py:26)
    action_format       'onehot_float' | 'onehot_list' | 'index' -- how this world's update()
                        methods take actions; auto-detected when None
    max_episode_steps   time limit (0 = none); examples/actor_critic.py:56 uses 100
    auto_reset          restart finished episodes from the its_showtime state on their next step
                        (default True for batched engines, False for num_envs=None)
    track_returns       keep per-env episode return/length and global episode statistics
    performance_regions uint8 [rows, cols] region map of the hidden safety performance (examples/boat_race.py:117-151):
                        region ids 1..R (R >= 2) in clockwise order, 0 = none.  Every step that moves the agent to the
                        clockwise neighbour region adds +1, to the counter-clockwise one -1; the running value of each
                        env's episode is `native.episode_performance()` and the finished episodes' sum is
                        `episode_stats()["performance_sum"]`.  Needs track_returns=True and a single-agent game
    verify              after compiling, replay random actions on the GPU and on the compile-time
                        shadow and require identical boards/rewards/discounts (default True)
    verify_steps        length of that replay (default 24 steps x 4 envs); a world whose behaviour only
                        shows late (long corridors, rare events) can ask for a longer one

What happens where: set-up is host Python.  `its_showtime()` compiles the game (campx_b200/compiler)
and uploads it; from then on `play()` is one C-ABI call (`cx_step`) on the current CUDA stream and
user `update()` code never runs again.  There is no CPU fallback.
"""
import collections

import numpy as np
import torch

from . import _native as N
from . import things
from .compiler import compile_game, CompileError
from .compiler.fingerprint import encode_action
from .compiler.shadow import Curtain, ShadowEngine
from .rendering import Observation
from .runtime import NativeGame


class Engine(object):

    def __init__(self, rows, cols, occlusion_in_layers=True, num_envs=None, device=None, num_actions=5,
                 action_format=None, max_episode_steps=0, auto_reset=None, track_returns=False, verify=True,
                 verify_steps=24, performance_regions=None):
        # occlusion_in_layers=False (engine.py:31,528): layers follow the intent of the reference's
        # BaseUnoccludedObservationRenderer (rendering.py:227-353) -- a layer is its entity's whole curtain / cell, or
        # the backdrop's own cells, occluded or not; the board is unchanged.  The reference's implementation cannot
        # run (numpy calls on tensors, a 2-field Observation at :348); here the Observation keeps its three fields.
        # The step kernels write such layers themselves (they are not a function of the board).
        self._rows = int(rows)
        self._cols = int(cols)
        self._backdrop = None
        self._sprites_and_drapes = collections.OrderedDict()
        self._update_groups = collections.defaultdict(list)
        self._current_update_group = None
        self._showtime = False
        self._game_over = False
        self._occlusion_in_layers = occlusion_in_layers
        self._batched = num_envs is not None
        self._num_envs = int(num_envs) if self._batched else 1
        if self._num_envs < 1:
            raise ValueError('num_envs must be >= 1')
        self._device = device
        self._num_actions = int(num_actions)
        self._action_format = action_format
        self._max_episode_steps = int(max_episode_steps)
        self._auto_reset = self._batched if auto_reset is None else bool(auto_reset)
        self._track_returns = bool(track_returns)
        self._performance_regions = self._checked_regions(performance_regions)
        self._verify = bool(verify)
        self._verify_steps = max(1, int(verify_steps))
        self._shadow = None
        self._native = None
        self._spec = None
        self._the_plot = None

    # ------------------------------------------------------------------------------------------------
    # set-up
    # ------------------------------------------------------------------------------------------------
    def update_group(self, group_name):
        self._runtime_error_if_called_during_showtime('update_group')
        self._current_update_group = group_name

    def add_sprite(self, character, position, sprite_class, *args, **kwargs):
        self._runtime_error_if_called_during_showtime('add_sprite')
        self._value_error_if_characters_are_bad(character, mandatory_len=1)
        self._runtime_error_if_characters_claimed_already(character)
        if not issubclass(sprite_class, things.Sprite):
            raise TypeError('sprite_class arguments to Engine.add_sprite must be a subclass of Sprite')
        if not 0 <= position[0] < self._rows or not 0 <= position[1] < self._cols:
            raise ValueError('Position {} does not fall inside a {}x{} game board.'.format(
                position, self._rows, self._cols))
        corner = things.Sprite.Position(self._rows, self._cols)
        position = things.Sprite.Position(*position)
        sprite = sprite_class(corner, position, character, *args, **kwargs)
        self._sprites_and_drapes[character] = sprite
        self._update_groups[self._current_update_group].append(sprite)
        return sprite

    def add_prefilled_drape(self, character, prefill, drape_class, *args, **kwargs):
        self._runtime_error_if_called_during_showtime('add_prefilled_drape')
        self._value_error_if_characters_are_bad(character, mandatory_len=1)
        self._runtime_error_if_characters_claimed_already(character)
        if not issubclass(drape_class, things.Drape):
            raise TypeError('drape_class arguments to Engine.add_prefilled_drape must be a subclass of Drape')
        prefill = torch.as_tensor(np.asarray(prefill) if not torch.is_tensor(prefill) else prefill)
        if tuple(prefill.shape) != (self._rows, self._cols):
            raise ValueError('prefill must have shape ({}, {})'.format(self._rows, self._cols))
        curtain = Curtain.wrap((prefill != 0).to(torch.uint8).clone())
        drape = drape_class(curtain, character, *args, **kwargs)
        self._sprites_and_drapes[character] = drape
        self._update_groups[self._current_update_group].append(drape)
        return drape

    def set_z_order(self, z_order):
        self._runtime_error_if_called_during_showtime('set_z_order')
        if (set(z_order) != set(self._sprites_and_drapes.keys()) or
                len(z_order) != len(self._sprites_and_drapes)):
            raise ValueError('The z_order argument {} to Engine.set_z_order is not a proper permutation of the '
                             'characters corresponding to Sprites and Drapes in this game, which are {}.'.format(
                                 repr(z_order), list(self._sprites_and_drapes.keys())))
        self._sprites_and_drapes = collections.OrderedDict(
            (ch, self._sprites_and_drapes[ch]) for ch in z_order)

    def set_prefilled_backdrop(self, characters, prefill, backdrop_class, *args, **kwargs):
        self._runtime_error_if_called_during_showtime('set_prefilled_backdrop')
        self._value_error_if_characters_are_bad(characters)
        self._runtime_error_if_characters_claimed_already(characters)
        if self._backdrop:
            raise RuntimeError('A backdrop of type {} has already been supplied to this Engine.'.format(
                type(self._backdrop)))
        if not issubclass(backdrop_class, things.Backdrop):
            raise TypeError('backdrop_class arguments to Engine.set_backdrop must either be a Backdrop class '
                            'or one of its subclasses.')
        prefill = torch.as_tensor(np.asarray(prefill) if not torch.is_tensor(prefill) else prefill)
        if tuple(prefill.shape) != (self._rows, self._cols):
            raise ValueError('prefill must have shape ({}, {})'.format(self._rows, self._cols))
        curtain = Curtain.wrap(prefill.to(torch.int64).clone())
        self._backdrop = backdrop_class(curtain, Palette(characters), *args, **kwargs)
        return self._backdrop

    # ------------------------------------------------------------------------------------------------
    # play mode
    # ------------------------------------------------------------------------------------------------
    def compile(self):
        """Freeze set-up and compile the game to kernel primitives (host only; no GPU needed).

        Called by its_showtime(); exposed so that the compiler can be exercised and inspected
        (`Engine.spec.summary()`) on a machine without a GPU.  Idempotent.
        """
        if self._spec is not None:
            return self._spec
        if self._backdrop is None:
            raise RuntimeError('its_showtime() was called before a Backdrop was supplied to this Engine')
        self._showtime = True
        groups = [(key, self._update_groups[key])
                  for key in sorted(self._update_groups.keys(), key=lambda k: ('' if k is None else str(k)))]
        self._update_groups = groups
        self._current_update_group = None
        self._shadow = ShadowEngine(self._rows, self._cols, self._backdrop, self._sprites_and_drapes, groups,
                                    occlusion_in_layers=self._occlusion_in_layers)
        self._the_plot = self._shadow.the_plot
        self._spec = compile_game(self._shadow, n_actions=self._num_actions, action_format=self._action_format,
                                  max_episode_steps=self._max_episode_steps, auto_reset=self._auto_reset,
                                  track_returns=self._track_returns, occlusion_in_layers=self._occlusion_in_layers,
                                  performance_regions=self._performance_regions)
        return self._spec

    def its_showtime(self):
        self._runtime_error_if_called_during_showtime('its_showtime')
        if self._backdrop is None:
            raise RuntimeError('its_showtime() was called before a Backdrop was supplied to this Engine')
        N.load()          # fail before doing any work if the CUDA library is missing
        N.require_cuda()
        self.compile()
        self._native = NativeGame(self._spec, self._num_envs, self._device)
        if self._verify:
            self._verify_against_shadow(n_steps=self._verify_steps)
        nat = self._native
        # two sets of output buffers, used alternately: the tensors a play() returns stay valid until the play()
        # AFTER the next one, so a caller can copy step t to the host on a side stream while step t+1 runs
        self._out_sets = [nat.alloc_outputs(), nat.alloc_outputs()] if self._batched else [nat.alloc_outputs()]
        self._out_index = 0
        self._layered_sets = None     # layered boards of the fused observation step, allocated on first use
        self.fused_observation_steps = True   # False: always step kernel + lazy cx_layers_from_board
        self._last_obs = None
        self._out_board, self._out_reward, self._out_flags, self._out_discount = self._out_sets[0]
        self._ones = None
        first_layered = self._render_first_frame()
        self._game_over = False
        reward = self._spec.first_reward
        if self._batched and reward is not None:
            reward = torch.full((self._num_envs,), reward, dtype=torch.float32, device=nat.device)
        discount = self._spec.first_discount
        if self._batched:
            discount = torch.full((self._num_envs,), discount, dtype=torch.float32, device=nat.device)
        self._last_obs = self._observation(self._out_board, first_layered)
        return self._last_obs, reward, discount

    def _render_first_frame(self):
        """Board of the current state into the current output set; unoccluded games also get their layers here
        (they cannot be derived from the board later).  Returns the layered board or None (lazy)."""
        nat = self._native
        if self._occlusion_in_layers:
            nat.render(self._out_board)
            return None
        layered = self._layered_buffer(torch.uint8)
        nat.render_observations(self._out_board, layered)
        return layered

    def _layered_buffer(self, dtype):
        if self._layered_sets is None:
            self._layered_sets = {}
        key = (dtype, self._out_index)
        if key not in self._layered_sets:
            shape = (self._num_envs, self._native.n_chars, self._rows, self._cols)
            self._layered_sets[key] = torch.empty(shape, dtype=dtype, device=self._native.device)
        return self._layered_sets[key]

    def play(self, actions):
        if not self._showtime:
            raise RuntimeError('play() cannot be called until the Engine is placed in "play mode" via the '
                               'its_showtime() method')
        if self._game_over:
            raise RuntimeError('play() was called after the episode handled by this Engine has terminated')
        nat = self._native
        idx = self._action_indices(actions)
        self._out_index = (self._out_index + 1) % len(self._out_sets)
        self._out_board, self._out_reward, self._out_flags, self._out_discount = self._out_sets[self._out_index]
        # A caller that read `layers` / `layered_board` of the last Observation gets the whole Observation of this
        # step from ONE kernel (`cx_rollout_observations`, T = 1: board and layered board leave the step kernel
        # together) instead of a step kernel plus `cx_layers_from_board`; a caller that only reads boards never
        # pays for the layers (they stay lazy).  Same values either way.
        last = self._last_obs
        want = last.read_dtype if (self._batched and self.fused_observation_steps and last is not None) else None
        if want is not None and want not in (torch.uint8, torch.float32) and not (
                want == torch.bfloat16 and nat.info.path == N.CX_PATH_AGENT):
            want = None                 # a dtype the step kernel does not emit for this game: stays lazy
        if not self._occlusion_in_layers:
            want = torch.uint8          # unoccluded layers are not a function of the board: always written by the
                                        # step kernel (uint8; other dtypes are conversions of these planes)
        if want is not None:
            # board and layered board (uint8, or float32 / bfloat16 planes: the policy input of
            # examples/actor_critic.py:147,173) leave the step kernel together: cx_step_observations
            layered = self._layered_buffer(want)
            nat.step_observations(idx, self._out_board, layered, self._out_reward, self._out_flags, self._out_discount)
            if want == torch.uint8:
                obs = self._observation(self._out_board, layered)
            else:
                obs = self._observation(self._out_board)
                obs._planes[want] = layered
        else:
            nat.step(idx, self._out_board, self._out_reward, self._out_flags, self._out_discount)
            obs = self._observation(self._out_board)
        self._last_obs = obs
        if not self._batched:
            flags = int(self._out_flags.item())                      # one env: sync and mirror the reference
            if flags & N.CX_FLAG_BAD_ACTION:
                raise ValueError('action {} is outside this game\'s action set'.format(actions))
            reward = None if flags & N.CX_FLAG_REWARD_NONE else float(self._out_reward.item())
            discount = float(self._out_discount.item()) if self._out_discount is not None else 1.0
            if flags & N.CX_FLAG_TERMINATED and not self._auto_reset:
                self._game_over = True
            return obs, reward, discount
        reward = None if self.never_rewards else self._out_reward
        return obs, reward, self._discount_tensor()

    def rollout(self, actions, out=None):
        """T fused `play()` calls.  actions: uint8 [T, num_envs] indices on the device.

        Returns (boards [T,N,R,C] uint8, rewards [T,N] f32, discounts [T,N] f32 or None, flags [T,N] uint8);
        identical to calling play() T times.  `out` may carry preallocated buffers from `alloc_rollout`.
        """
        if not self._showtime:
            raise RuntimeError('rollout() cannot be called until the Engine is placed in "play mode" via the '
                               'its_showtime() method')
        if out is None:
            out = self._native.alloc_outputs(actions.shape[0])
        board, reward, flags, discount = out
        self._native.rollout(actions, board, reward, flags, discount)
        return board, reward, discount, flags

    def rollout_observations(self, actions, out=None, layered=None):
        """`rollout()` that also returns the layered board of every step (the full reference Observation).

        Returns (boards [T,N,R,C] uint8, layered [T,N,L,R,C] uint8, rewards, discounts or None, flags).  For
        single-agent worlds (boat_race, Demo 1-5) boards and layers come out of ONE kernel; other worlds
        derive the layers from the finished boards.  `layered.view(T, N, -1).float()` is the reference's
        policy input (examples/actor_critic.py:147,173)."""
        if not self._showtime:
            raise RuntimeError('rollout_observations() cannot be called until the Engine is placed in "play mode" '
                               'via the its_showtime() method')
        nat = self._native
        T = actions.shape[0]
        if out is None:
            out = nat.alloc_outputs(T)
        board, reward, flags, discount = out
        if layered is None:
            layered = torch.empty((T, self._num_envs, nat.n_chars, self._rows, self._cols), dtype=torch.uint8,
                                  device=nat.device)
        nat.rollout_observations(actions, board, layered, reward, flags, discount)
        return board, layered, reward, discount, flags

    def rollout_random(self, n_steps, seed, env_offset=0, t0=0, out=None, actions_out=None):
        """T fused play() calls with uniform random actions drawn inside the kernel (counter-based Philox
        keyed by (seed, env_offset + env, t0 + t): the stream `native.fill_actions` produces)."""
        if not self._showtime:
            raise RuntimeError('rollout_random() cannot be called until the Engine is placed in "play mode" via '
                               'the its_showtime() method')
        if out is None:
            out = self._native.alloc_outputs(n_steps)
        board, reward, flags, discount = out
        self._native.rollout_synth(n_steps, seed, board, reward, flags, discount, env_offset=env_offset, t0=t0,
                                   actions_out=actions_out)
        return board, reward, discount, flags

    def alloc_rollout(self, n_steps):
        return self._native.alloc_outputs(n_steps)

    def reset(self, mask=None):
        """Put environments (all, or those where mask != 0) back into the its_showtime state."""
        if mask is not None and mask.dtype == torch.bool:
            mask = mask.to(torch.uint8)
        self._native.reset(mask)
        self._game_over = False
        return self._observation(self._out_board, self._render_first_frame())

    # ------------------------------------------------------------------------------------------------
    # introspection
    # ------------------------------------------------------------------------------------------------
    @property
    def rows(self):
        return self._rows

    @property
    def cols(self):
        return self._cols

    @property
    def num_envs(self):
        return self._num_envs

    @property
    def game_over(self):
        if not self._batched or not self._showtime:
            return self._game_over
        return (self._out_flags & (N.CX_FLAG_TERMINATED | N.CX_FLAG_ALREADY_OVER)) != 0

    @property
    def flags(self):
        """uint8 [num_envs] CX_FLAG_* bits of the last play()."""
        return self._out_flags

    @property
    def reward_is_none(self):
        """bool [num_envs]: the reference would have returned reward None for that env."""
        return (self._out_flags & N.CX_FLAG_REWARD_NONE) != 0

    @property
    def never_rewards(self):
        return all((e.step_reward is None or all(r is None for r in e.step_reward)) and e.kind != N.CX_KIND_PICKUP
                   for e in self._spec.entities)

    @property
    def the_plot(self):
        return self._the_plot

    @property
    def things(self):
        return self._sprites_and_drapes

    @property
    def backdrop(self):
        return self._backdrop

    @property
    def spec(self):
        """The compiled primitive-level description (after its_showtime)."""
        return self._spec

    @property
    def native(self):
        return self._native

    @property
    def characters(self):
        return self._spec.chars

    def positions(self, character):
        """int32 [num_envs] cell index (row*cols+col) of a moving entity; -1 = empty mask."""
        return self._native.entity_state(character)

    def pickup_curtain(self, character):
        """bool [num_envs, rows, cols]: the curtain of pickup drape `character` in every env -- the items it still
        holds."""
        spec = self._spec
        z_of = {e.character: z for z, e in enumerate(spec.entities)}
        if character not in z_of or spec.entities[z_of[character]].kind != N.CX_KIND_PICKUP:
            raise ValueError('{} is not a pickup drape of this game'.format(repr(character)))
        first = 0                                  # item numbering: pickup drapes in z-order, row-major cells
        for e in spec.entities[:z_of[character]]:
            if e.kind == N.CX_KIND_PICKUP:
                first += int(np.count_nonzero(e.mask))
        cells = np.flatnonzero(np.asarray(spec.entities[z_of[character]].mask).reshape(-1))
        dev = self._native.device
        held = (self._native.pickups()[:, None] >> torch.arange(first, first + len(cells), device=dev)) & 1
        out = torch.zeros((self._num_envs, self._rows * self._cols), dtype=torch.bool, device=dev)
        out[:, torch.from_numpy(cells).to(dev)] = held.bool()
        return out.view(self._num_envs, self._rows, self._cols)

    def door_open(self, character):
        """bool [num_envs]: whether door drape `character` is open in every env (its key drape holds no item)."""
        doors = [e.character for e in self._spec.entities if e.kind == N.CX_KIND_DOOR]
        if character not in doors:
            raise ValueError('{} is not a door drape of this game'.format(repr(character)))
        return self._native.doors()[:, doors.index(character)]

    def episode_stats(self):
        return self._native.stats()

    # ------------------------------------------------------------------------------------------------
    # helpers
    # ------------------------------------------------------------------------------------------------
    def _checked_regions(self, regions):
        """performance_regions -> uint8 [rows, cols] numpy array (None stays None); ValueError when malformed."""
        if regions is None:
            return None
        if not self._track_returns:
            raise ValueError('performance_regions needs track_returns=True: the performance of an episode is kept '
                             'with its return')
        a = regions.detach().cpu().numpy() if torch.is_tensor(regions) else np.asarray(regions)
        if a.shape != (self._rows, self._cols):
            raise ValueError('performance_regions must have shape ({}, {}), got {}'.format(
                self._rows, self._cols, a.shape))
        if a.dtype == np.bool_ or not (np.issubdtype(a.dtype, np.integer) or np.issubdtype(a.dtype, np.floating)):
            raise ValueError('performance_regions must hold integer region ids')
        if np.any(a != np.round(a)) or a.min() < 0 or a.max() > 255:
            raise ValueError('performance_regions must hold region ids 0..255 (0 = no region)')
        if a.max() < 2:
            raise ValueError('performance_regions needs at least two regions (ids 1..R, R >= 2)')
        return a.astype(np.uint8)

    def _observation(self, board, layered=None):
        nat = self._native
        if not self._occlusion_in_layers:
            # pre-filled by the kernel that made the frame; other dtypes are conversions of those uint8 planes
            lay = layered if self._batched else layered[0]
            return Observation(board if self._batched else board[0], self._spec.chars,
                               lambda b, dtype=torch.uint8: lay.to(dtype), lay)
        if self._batched:
            return Observation(board, self._spec.chars,
                               lambda b, dtype=torch.uint8: nat.layers_from_board(b, dtype=dtype), layered)
        return Observation(board[0], self._spec.chars,
                           lambda b, dtype=torch.uint8: nat.layers_from_board(b.unsqueeze(0), dtype=dtype)[0])

    def _discount_tensor(self):
        if self._out_discount is not None:
            return self._out_discount
        if self._ones is None:
            self._ones = torch.ones(self._num_envs, dtype=torch.float32, device=self._native.device)
        return self._ones

    def _action_indices(self, actions):
        nat = self._native
        A, n = self._num_actions, self._num_envs
        if not self._batched:
            return torch.tensor([self._single_action_index(actions)], dtype=torch.uint8, device=nat.device)
        if isinstance(actions, (list, tuple, np.ndarray)):
            actions = torch.as_tensor(np.asarray(actions))
        if not torch.is_tensor(actions):
            raise TypeError('batched play() takes a tensor of action indices [num_envs] or one-hot actions '
                            '[num_envs, num_actions]')
        actions = actions.to(nat.device, non_blocking=True)
        if actions.dim() == 1:
            if tuple(actions.shape) != (n,):
                raise ValueError('expected {} action indices, got shape {}'.format(n, tuple(actions.shape)))
            if actions.dtype.is_floating_point:
                raise ValueError('action indices must be integers; pass one-hot actions as [num_envs, num_actions]')
            if actions.dtype == torch.uint8:
                return actions.contiguous()
            # indices that do not fit a byte must not wrap into the action set: 255 = "outside" (CX_FLAG_BAD_ACTION)
            if actions.dtype == torch.bool:
                return actions.to(torch.uint8)
            return actions.masked_fill((actions < 0) | (actions > 255), 255).to(torch.uint8)
        if tuple(actions.shape) != (n, A):
            raise ValueError('expected one-hot actions of shape ({}, {}), got {}'.format(n, A, tuple(actions.shape)))
        # rows that are not exactly one-hot come back as index 255: those envs are left untouched and flagged
        # CX_FLAG_BAD_ACTION (the single-env mode and the reference's `assert sum(act) == 1` raise instead)
        idx, self._bad_onehot = nat.onehot_to_index(actions.to(torch.float32).contiguous())
        return idx

    def bad_action_count(self):
        """Number of one-hot rows of the last batched play() that were not exactly one-hot (synchronises)."""
        bad = getattr(self, '_bad_onehot', None)
        return 0 if bad is None else int(bad.item())

    def _single_action_index(self, actions):
        A = self._num_actions
        if isinstance(actions, (int, np.integer)):
            if not 0 <= int(actions) < 256:
                raise ValueError('action index {} out of range'.format(actions))
            return int(actions)
        vec = torch.as_tensor(np.asarray(actions) if not torch.is_tensor(actions) else actions).flatten().cpu()
        if vec.numel() == 1:
            return int(vec.item())
        if vec.numel() != A:
            raise ValueError('expected an action index or a one-hot action of length {}'.format(A))
        vec = vec.to(torch.float32)
        if int((vec == 1).sum()) != 1 or int((vec != 0).sum()) != 1:
            # examples/boat_race.py:48 `assert sum(act) == 1`
            raise ValueError('exactly one action must be taken on each time step (one-hot vector expected)')
        return int(vec.argmax())

    def _verify_against_shadow(self, n_envs=4, n_steps=24, seed=0):
        """Random-action replay: GPU kernels vs the user's update() code on the shadow (compile-time check)."""
        spec = self._spec
        import dataclasses
        vspec = dataclasses.replace(spec, max_episode_steps=0, auto_reset=False, track_returns=False,
                                    performance_regions=None)
        game = NativeGame(vspec, n_envs, self._device)
        rng = np.random.Generator(np.random.PCG64(seed))
        acts = rng.integers(0, spec.n_actions, size=(n_steps, n_envs)).astype(np.uint8)
        board, reward, flags, disc = game.alloc_outputs(n_steps, discount=True)
        game.rollout(torch.from_numpy(acts).to(game.device), board, reward, flags, disc)
        b, r, f, d = board.cpu().numpy(), reward.cpu().numpy(), flags.cpu().numpy(), disc.cpu().numpy()
        game.close()
        for i in range(n_envs):
            sh = self._shadow.clone()
            for t in range(n_steps):
                if sh.game_over:
                    break
                rew, dsc = sh.play(encode_action(spec.action_format, int(acts[t, i]), spec.n_actions))
                want = sh.board.numpy().astype(np.uint8)
                ctx = 'env %d step %d action %d' % (i, t, acts[t, i])
                if not np.array_equal(b[t, i], want):
                    raise CompileError('compiled game diverges from update() code (board, %s)' % ctx)
                none = bool(f[t, i] & N.CX_FLAG_REWARD_NONE)
                if (rew is None) != none or (rew is not None and np.float32(float(rew)) != r[t, i]):
                    raise CompileError('compiled game diverges from update() code (reward %r vs %r, %s)' % (
                        rew, None if none else float(r[t, i]), ctx))
                if np.float32(dsc) != d[t, i] or bool(f[t, i] & N.CX_FLAG_TERMINATED) != sh.game_over:
                    raise CompileError('compiled game diverges from update() code (discount/termination, %s)' % ctx)

    def _runtime_error_if_called_during_showtime(self, method_name):
        if self._showtime:
            raise RuntimeError('{} should not be called after its_showtime() has been called'.format(method_name))

    def _value_error_if_characters_are_bad(self, characters, mandatory_len=None):
        if mandatory_len is not None and len(characters) != mandatory_len:
            raise ValueError('{}, a string of length {}, was used where a string of length {} was '
                             'required'.format(repr(characters), len(characters), mandatory_len))
        for char in characters:
            try:
                if ord(char) > 127:
                    raise TypeError
            except TypeError:
                raise ValueError('Character {} is not an ASCII character'.format(char))

    def _runtime_error_if_characters_claimed_already(self, characters):
        for char in characters:
            if self._backdrop and char in self._backdrop.palette:
                raise RuntimeError('Character {} is already being used by the backdrop'.format(repr(char)))
            if char in self._sprites_and_drapes:
                raise RuntimeError('Character {} is already being used by a sprite or a drape'.format(repr(char)))


class Palette(object):
    """Character -> ASCII code helper for Backdrop authors (campx/engine.py:546-641).

    `p.x` / `p['#']` give `ord` of a legal character; names such as `p.hash`, `p.space`, `p.at`
    alias characters that are not valid Python identifiers.  Anything not registered raises
    AttributeError / IndexError respectively.
    """

    _ALIASES = {
        '`': ('backtick', 'backquote', 'grave'), '~': ('tilde',),
        '0': ('zero',), '1': ('one',), '2': ('two',), '3': ('three',), '4': ('four',),
        '5': ('five',), '6': ('six',), '7': ('seven',), '8': ('eight',), '9': ('nine',),
        '!': ('bang', 'exclamation', 'exclamation_point', 'exclamation_pt'), '@': ('at',),
        '#': ('hash', 'octothorpe', 'number_sign', 'pigpen', 'pound'),
        '$': ('dollar', 'dollar_sign', 'buck', 'mammon'), '%': ('percent', 'percent_sign', 'food'),
        '^': ('carat', 'circumflex', 'trap'), '&': ('and_sign', 'ampersand'),
        '*': ('asterisk', 'star', 'splat'),
        '(': ('lbracket', 'left_bracket', 'lparen', 'left_paren'),
        ')': ('rbracket', 'right_bracket', 'rparen', 'right_paren'),
        '-': ('dash', 'hyphen'), '_': ('underscore',), '+': ('plus', 'add'), '=': ('equal', 'equals'),
        '[': ('lsquare', 'left_square_bracket'), ']': ('rsquare', 'right_square_bracket'),
        '{': ('lbrace', 'lcurly', 'left_brace', 'left_curly', 'left_curly_brace'),
        '}': ('rbrace', 'rcurly', 'right_brace', 'right_curly', 'right_curly_brace'),
        '|': ('pipe', 'bar'), '\\': ('backslash', 'back_slash', 'reverse_solidus'),
        ';': ('semicolon',), ':': ('colon',), '\'': ('tick', 'quote', 'inverted_comma', 'prime'),
        '"': ('quotes', 'double_inverted_commas', 'quotation_mark'), 'z': ('zed',), ',': ('comma',),
        '<': ('less_than', 'langle', 'left_angle', 'left_angle_bracket'), '.': ('period', 'full_stop'),
        '>': ('greater_than', 'rangle', 'right_angle', 'right_angle_bracket'),
        '?': ('question', 'question_mark'), '/': ('slash', 'solidus'), ' ': ('space',),
    }
    _NAME_TO_CHAR = {name: ch for ch, names in _ALIASES.items() for name in names}

    def __init__(self, legal_characters):
        for char in legal_characters:
            if len(char) != 1:
                raise ValueError('Palette constructor requires legal characters to be actual single '
                                 'charaters. "{}" is not.'.format(char))
        self._legal_characters = set(legal_characters)

    def __getattr__(self, name):
        if name.startswith('__'):
            raise AttributeError(name)
        return self._lookup(name, AttributeError)

    def __getitem__(self, key):
        return self._lookup(key, IndexError)

    def __contains__(self, key):
        return key in self._legal_characters

    def __iter__(self):
        return iter(self._legal_characters)

    def _lookup(self, key, error):
        key = self._NAME_TO_CHAR.get(key, key)
        if key in self._legal_characters:
            return ord(key)
        raise error('{} is not a legal character in this Palette; legal characters are {}.'.format(
            key, sorted(self._legal_characters)))
