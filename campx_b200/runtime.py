"""Device runtime: owns the native game handle, the per-env state blob and the output buffers, and
issues the C-ABI calls on the current torch CUDA stream.

PyTorch is plumbing here (device memory, streams); every byte of simulation work happens inside
libcampx_b200.so.  Nothing in this module has a CPU code path.
"""
import ctypes

import torch

from . import _native as N
from .description import GameSpec


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class NativeGame(object):
    """A compiled game resident on one GPU for `num_envs` environments."""

    def __init__(self, spec: GameSpec, num_envs: int, device=None):
        N.require_cuda()
        self._lib = N.load()
        self.spec = spec
        self.num_envs = int(num_envs)
        if self.num_envs < 1:
            raise ValueError("num_envs must be >= 1")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise N.NativeLibraryError("campx_b200 runs on CUDA devices only (got %s)" % self.device)
        self._handle = ctypes.c_void_p()
        desc, keep = spec.to_ctypes()
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_game_create(ctypes.byref(desc), ctypes.byref(self._handle)))
        del keep
        info = N.GameInfo()
        N.check(self._lib.cx_game_get_info(self._handle, ctypes.byref(info)))
        self.info = info
        self.rows, self.cols, self.cells = info.rows, info.cols, info.cells
        self.n_chars, self.n_actions = info.n_chars, info.n_actions
        self.can_terminate = bool(info.can_terminate)
        self.tracks = bool(info.tracks)
        self.tracks_performance = bool(info.tracks_performance)
        nbytes = self._lib.cx_state_bytes(self._handle, self.num_envs)
        if nbytes <= 0:
            raise RuntimeError("cx_state_bytes failed")
        self.state = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        assert self.state.data_ptr() % 256 == 0
        self._z_of = {e.character: z for z, e in enumerate(spec.entities)}
        self.reset()

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_handle", None) is not None and self._handle.value:
            self._lib.cx_game_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- buffers --------------------------------------------------------------------------------------
    def alloc_outputs(self, n_steps=None, discount=None):
        """Allocate (board, reward, flags, discount) for one step ([n,...]) or a rollout ([T,n,...])."""
        lead = (self.num_envs,) if n_steps is None else (int(n_steps), self.num_envs)
        want_discount = self.wants_discount if discount is None else discount
        board = torch.empty(lead + (self.rows, self.cols), dtype=torch.uint8, device=self.device)
        reward = torch.empty(lead, dtype=torch.float32, device=self.device)
        flags = torch.empty(lead, dtype=torch.uint8, device=self.device)
        disc = torch.empty(lead, dtype=torch.float32, device=self.device) if want_discount else None
        return board, reward, flags, disc

    @property
    def wants_discount(self):
        """Discount is only materialised when some action can change it (terminate / default discount)."""
        return self.can_terminate or any(e.discount for e in self.spec.entities)

    # -- C-ABI calls --------------------------------------------------------------------------------------
    def reset(self, mask=None):
        if mask is not None:
            mask = self._check(mask, torch.uint8, (self.num_envs,), "mask")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_reset(self._handle, _ptr(self.state), self.num_envs, _ptr(mask), _stream()))

    def render(self, board=None):
        if board is None:
            board = torch.empty((self.num_envs, self.rows, self.cols), dtype=torch.uint8, device=self.device)
        self._check(board, torch.uint8, (self.num_envs, self.rows, self.cols), "board")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_render(self._handle, _ptr(self.state), self.num_envs, _ptr(board), _stream()))
        return board

    def step(self, actions, board, reward, flags, discount=None):
        n = self.num_envs
        self._check(actions, torch.uint8, (n,), "actions")
        self._check(board, torch.uint8, (n, self.rows, self.cols), "board")
        self._check(reward, torch.float32, (n,), "reward")
        self._check(flags, torch.uint8, (n,), "flags")
        if discount is not None:
            self._check(discount, torch.float32, (n,), "discount")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_step(self._handle, _ptr(self.state), n, _ptr(actions), _ptr(reward),
                                      _ptr(discount), _ptr(flags), _ptr(board), _stream()))

    def rollout(self, actions, board, reward, flags, discount=None):
        n = self.num_envs
        if actions.dim() != 2:
            raise ValueError("rollout actions must be [T, num_envs]")
        T = actions.shape[0]
        self._check(actions, torch.uint8, (T, n), "actions")
        self._check(board, torch.uint8, (T, n, self.rows, self.cols), "board")
        self._check(reward, torch.float32, (T, n), "reward")
        self._check(flags, torch.uint8, (T, n), "flags")
        if discount is not None:
            self._check(discount, torch.float32, (T, n), "discount")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_rollout(self._handle, _ptr(self.state), n, T, _ptr(actions), _ptr(reward),
                                         _ptr(discount), _ptr(flags), _ptr(board), _stream()))

    def rollout_observations(self, actions, board, layered, reward, flags, discount=None):
        """Fused rollout that writes the layered board [T, n, n_chars, rows, cols] next to every board."""
        n = self.num_envs
        if actions.dim() != 2:
            raise ValueError("rollout actions must be [T, num_envs]")
        T = actions.shape[0]
        self._check(actions, torch.uint8, (T, n), "actions")
        self._check(board, torch.uint8, (T, n, self.rows, self.cols), "board")
        self._check(layered, torch.uint8, (T, n, self.n_chars, self.rows, self.cols), "layered")
        self._check(reward, torch.float32, (T, n), "reward")
        self._check(flags, torch.uint8, (T, n), "flags")
        if discount is not None:
            self._check(discount, torch.float32, (T, n), "discount")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_rollout_observations(self._handle, _ptr(self.state), n, T, _ptr(actions),
                                                      _ptr(reward), _ptr(discount), _ptr(flags), _ptr(board),
                                                      _ptr(layered), _stream()))

    _DTYPES = {torch.uint8: N.CX_DTYPE_U8, torch.float32: N.CX_DTYPE_F32, torch.bfloat16: N.CX_DTYPE_BF16}

    def step_observations(self, actions, board, layered, reward, flags, discount=None):
        """One play() that also writes the layered board [n, n_chars, rows, cols] as uint8, float32 or bfloat16
        (the policy input of examples/actor_critic.py:147,173) from the step kernel itself."""
        n = self.num_envs
        self._check(actions, torch.uint8, (n,), "actions")
        self._check(board, torch.uint8, (n, self.rows, self.cols), "board")
        if not isinstance(layered, torch.Tensor) or layered.dtype not in self._DTYPES:
            raise ValueError("layered must be a uint8, float32 or bfloat16 tensor")
        if layered.numel() != n * self.n_chars * self.cells:
            raise ValueError("layered must hold %d x %d x %d elements (got shape %s)"
                             % (n, self.n_chars, self.cells, tuple(layered.shape)))
        self._check(layered, layered.dtype, tuple(layered.shape), "layered")
        self._check(reward, torch.float32, (n,), "reward")
        self._check(flags, torch.uint8, (n,), "flags")
        if discount is not None:
            self._check(discount, torch.float32, (n,), "discount")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_step_observations(self._handle, _ptr(self.state), n, _ptr(actions), _ptr(reward),
                                                   _ptr(discount), _ptr(flags), _ptr(board), _ptr(layered),
                                                   self._DTYPES[layered.dtype], _stream()))

    def render_observations(self, board, layered):
        """The frame of the CURRENT state with its layered board (first Observation / after a reset); no step."""
        n = self.num_envs
        self._check(board, torch.uint8, (n, self.rows, self.cols), "board")
        if not isinstance(layered, torch.Tensor) or layered.dtype not in self._DTYPES:
            raise ValueError("layered must be a uint8, float32 or bfloat16 tensor")
        self._check(layered, layered.dtype, (n, self.n_chars, self.rows, self.cols), "layered")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_render_observations(self._handle, _ptr(self.state), n, _ptr(board), _ptr(layered),
                                                     self._DTYPES[layered.dtype], _stream()))

    def sample_actions(self, scores, seed, step=None, step_offset=0, logits=False, env_offset=0, out=None, logp=None):
        """Categorical(probs).sample() for every env (examples/actor_critic.py:90-98) -> uint8 [n] action indices.

        scores: float32 [n, n_actions] probabilities (or logits with logits=True).  The uniform numbers come from
        the Philox stream (seed; env_offset + env, step), step = step[0] + step_offset where `step` is an optional
        int64 device tensor -- a captured CUDA graph advances it between replays."""
        n = self.num_envs
        self._check(scores, torch.float32, (n, self.n_actions), "scores")
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=self.device)
        self._check(out, torch.uint8, (n,), "actions")
        if step is not None:
            self._check(step, torch.int64, (1,), "step")
        if logp is not None:
            self._check(logp, torch.float32, (n,), "logp")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_sample_actions(_ptr(scores), n, self.n_actions, 1 if logits else 0, int(seed),
                                                int(env_offset), _ptr(step), int(step_offset), _ptr(out), _ptr(logp),
                                                _stream()))
        return out

    def policy_sample(self, x, w1t, b1, w2, b2, seed, step=None, step_offset=0, env_offset=0, out=None, logp=None,
                      logits_out=None):
        """relu(x @ w1t + b1) @ w2.T + b2 -> softmax -> Categorical.sample() in ONE launch: the acting half of the
        reference's Policy (examples/actor_critic.py:64-98) -> uint8 [n] action indices.  x float32 [n, n_inputs]
        (e.g. the planes step_observations wrote); w1t [n_inputs, n_hidden] is affine1.weight TRANSPOSED
        (`weight.t().contiguous()`), w2 / b1 / b2 in torch.nn.Linear layout; n_hidden <= 32.  Sampling as in
        sample_actions(logits=True): equal logits give equal actions."""
        n = self.num_envs
        if x.dim() != 2 or x.shape[0] != n or w1t.dim() != 2:
            raise ValueError("x must be [num_envs, n_inputs], w1t [n_inputs, n_hidden]")
        n_in, n_hidden = int(x.shape[1]), int(w1t.shape[1])
        self._check(x, torch.float32, (n, n_in), "x")
        self._check(w1t, torch.float32, (n_in, n_hidden), "w1t")
        self._check(b1, torch.float32, (n_hidden,), "b1")
        self._check(w2, torch.float32, (self.n_actions, n_hidden), "w2")
        self._check(b2, torch.float32, (self.n_actions,), "b2")
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=self.device)
        self._check(out, torch.uint8, (n,), "actions")
        if step is not None:
            self._check(step, torch.int64, (1,), "step")
        if logp is not None:
            self._check(logp, torch.float32, (n,), "logp")
        if logits_out is not None:
            self._check(logits_out, torch.float32, (n, self.n_actions), "logits_out")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_policy_sample(_ptr(x), n, n_in, _ptr(w1t), _ptr(b1), n_hidden, _ptr(w2), _ptr(b2),
                                               self.n_actions, int(seed), int(env_offset), _ptr(step), int(step_offset),
                                               _ptr(out), _ptr(logp), _ptr(logits_out), _stream()))
        return out

    def policy_sample_board(self, board, w1t, b1, w2, b2, seed, step=None, step_offset=0, env_offset=0, out=None,
                            logp=None, logits_out=None):
        """policy_sample on the layered board of `board` as float32 planes (examples/actor_critic.py:147,173), read off
        the uint8 board itself: the planes are never written.  board uint8 [num_envs, rows, cols] (e.g. one step of a
        [T + 1, num_envs, rows, cols] rollout buffer); w1t [n_chars * cells, n_hidden] is affine1.weight TRANSPOSED.
        Any board size, single-agent and generic games; occluded layers only (NotImplementedError otherwise).  For
        finite weights: the bits of policy_sample(layers_from_board(board, dtype=float32).view(num_envs, -1), ...)."""
        n, feat = self.num_envs, self.n_chars * self.cells
        self._check(board, torch.uint8, (n, self.rows, self.cols), "board")
        if w1t.dim() != 2:
            raise ValueError("w1t must be [n_chars * cells, n_hidden]")
        n_hidden = int(w1t.shape[1])
        self._check(w1t, torch.float32, (feat, n_hidden), "w1t")
        self._check(b1, torch.float32, (n_hidden,), "b1")
        self._check(w2, torch.float32, (self.n_actions, n_hidden), "w2")
        self._check(b2, torch.float32, (self.n_actions,), "b2")
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=self.device)
        self._check(out, torch.uint8, (n,), "actions")
        if step is not None:
            self._check(step, torch.int64, (1,), "step")
        if logp is not None:
            self._check(logp, torch.float32, (n,), "logp")
        if logits_out is not None:
            self._check(logits_out, torch.float32, (n, self.n_actions), "logits_out")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_policy_sample_board(self._handle, _ptr(board), n, _ptr(w1t), _ptr(b1), n_hidden,
                                                     _ptr(w2), _ptr(b2), int(seed), int(env_offset), _ptr(step),
                                                     int(step_offset), _ptr(out), _ptr(logp), _ptr(logits_out),
                                                     _stream()))
        return out

    def rollout_policy(self, n_steps, w1t, b1, w2, b2, seed, states, actions, reward, flags, step=None, step_offset=0,
                       env_offset=0, logp=None):
        """The reference's actor-critic rollout loop (examples/actor_critic.py:146-173) in ONE launch: T times
        (policy -> sample -> play), bit-identical to T x (policy_sample + step_observations(float32)).
        states float32 [T + 1, n, n_chars * cells]: states[t] = policy input before action t (states[0]: now)."""
        n, T, feat = self.num_envs, int(n_steps), self.n_chars * self.cells
        n_hidden = int(w1t.shape[1])
        self._check(w1t, torch.float32, (feat, n_hidden), "w1t")
        self._check(b1, torch.float32, (n_hidden,), "b1")
        self._check(w2, torch.float32, (self.n_actions, n_hidden), "w2")
        self._check(b2, torch.float32, (self.n_actions,), "b2")
        self._check(states, torch.float32, (T + 1, n, feat), "states")
        self._check(actions, torch.uint8, (T, n), "actions")
        self._check(reward, torch.float32, (T, n), "reward")
        self._check(flags, torch.uint8, (T, n), "flags")
        if step is not None:
            self._check(step, torch.int64, (1,), "step")
        if logp is not None:
            self._check(logp, torch.float32, (T, n), "logp")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_rollout_policy(self._handle, _ptr(self.state), n, T, _ptr(w1t), _ptr(b1), n_hidden,
                                                _ptr(w2), _ptr(b2), int(seed), int(env_offset), _ptr(step),
                                                int(step_offset), _ptr(states), _ptr(actions), _ptr(reward), _ptr(flags),
                                                _ptr(logp), _stream()))

    def rollout_synth(self, n_steps, seed, board, reward, flags, discount=None, env_offset=0, t0=0, actions_out=None):
        """Fused rollout with uniform random actions generated inside the kernel (no action bytes read);
        identical to fill_actions(seed, env_offset, t0) + rollout."""
        n, T = self.num_envs, int(n_steps)
        self._check(board, torch.uint8, (T, n, self.rows, self.cols), "board")
        self._check(reward, torch.float32, (T, n), "reward")
        self._check(flags, torch.uint8, (T, n), "flags")
        if discount is not None:
            self._check(discount, torch.float32, (T, n), "discount")
        if actions_out is not None:
            self._check(actions_out, torch.uint8, (T, n), "actions_out")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_rollout_synth(self._handle, _ptr(self.state), n, T, int(seed), int(env_offset),
                                               int(t0), _ptr(actions_out), _ptr(reward), _ptr(discount),
                                               _ptr(flags), _ptr(board), _stream()))

    def layers_from_board(self, board, out=None, dtype=torch.uint8):
        """[..., rows, cols] boards -> [..., n_chars, rows, cols] layered boards (rendering.py:204-215)."""
        if board.dtype != torch.uint8 or not board.is_contiguous() or board.device != self.device:
            raise ValueError("board must be a contiguous uint8 tensor on %s" % self.device)
        lead = tuple(board.shape[:-2])
        nb = 1
        for s in lead:
            nb *= s
        shape = lead + (self.n_chars, self.rows, self.cols)
        if out is None:
            out = torch.empty(shape, dtype=dtype, device=self.device)
        self._check(out, dtype, shape, "layered")
        fn = self._lib.cx_layers_from_board if dtype == torch.uint8 else self._lib.cx_layers_from_board_f32
        if dtype not in (torch.uint8, torch.float32):
            raise ValueError("layered dtype must be uint8 or float32")
        with torch.cuda.device(self.device):
            N.check(fn(self._handle, _ptr(board), nb, _ptr(out), _stream()))
        return out

    def onehot_to_index(self, onehot, out=None):
        n = self.num_envs
        self._check(onehot, torch.float32, (n, self.n_actions), "one-hot actions")
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=self.device)
        bad = torch.zeros(1, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_onehot_to_index(_ptr(onehot), n, self.n_actions, _ptr(out), _ptr(bad), _stream()))
        return out, bad

    def fill_actions(self, n_steps, seed, env_offset=0, t0=0, out=None):
        """Synthetic uniform actions [T, n] from counter-based Philox (seed, env_offset+i, t0+t)."""
        if out is None:
            out = torch.empty((int(n_steps), self.num_envs), dtype=torch.uint8, device=self.device)
        self._check(out, torch.uint8, (int(n_steps), self.num_envs), "actions")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_fill_actions(int(seed), int(env_offset), int(t0), int(n_steps), self.num_envs,
                                              self.n_actions, _ptr(out), _stream()))
        return out

    def entity_state(self, character):
        out = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_get_entity_state(self._handle, _ptr(self.state), self.num_envs,
                                                  self._z_of[character], _ptr(out), _stream()))
        return out

    def set_entity_state(self, character, cells):
        cells = self._check(cells, torch.int32, (self.num_envs,), "cells")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_set_entity_state(self._handle, _ptr(self.state), self.num_envs,
                                                  self._z_of[character], _ptr(cells), _stream()))

    def render_state(self):
        """(z_order uint32 [N]: 4 bits per z position back to front = entity id, visible uint32 [N]: bit z,
        backdrop_offset int32 [N]: row * cols + col) -- the render state of games where it changes during play."""
        z = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        vis = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        off = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_get_render_state(self._handle, _ptr(self.state), self.num_envs, _ptr(z), _ptr(vis),
                                                  _ptr(off), _stream()))
        return z, vis, off

    def episode_state(self):
        steps = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        returns = torch.empty(self.num_envs, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_get_episode_state(self._handle, _ptr(self.state), self.num_envs, _ptr(steps),
                                                   _ptr(returns), _stream()))
        return steps, returns

    def episode_performance(self):
        """float32 [num_envs] running safety performance of every env's current episode (games created with
        performance_regions)."""
        perf = torch.empty(self.num_envs, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_get_episode_performance(self._handle, _ptr(self.state), self.num_envs, _ptr(perf),
                                                         _stream()))
        return perf

    def pickups(self):
        """int64 [num_envs]: bit i set = item i is still on the board (games with pickup drapes).  Items are numbered
        pickup drape by pickup drape in z-order, row-major within a drape (`Engine.pickup_curtain` unpacks them)."""
        bits = torch.empty(self.num_envs, dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_get_pickups(self._handle, _ptr(self.state), self.num_envs, _ptr(bits), _stream()))
        return bits

    def fold_stats(self):
        """Add the kernels' partial statistics blocks into the float64[8] block at the head of the state blob
        (asynchronous on the current stream)."""
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_stats_fold(self._handle, _ptr(self.state), _stream()))

    @property
    def stats_tensor(self):
        """float64[8] view of the (folded) episode statistics inside the state blob.  The kernels keep adding to the
        blob, so all-reduce a CLONE over ranks (campx_b200.dist.all_reduce_stats), not the view itself -- a view that
        holds the global sums would be summed over ranks again at the next report."""
        self.fold_stats()
        return self.state[:8 * N.CX_STATS_DOUBLES].view(torch.float64)

    def stats(self):
        buf = (ctypes.c_double * N.CX_STATS_DOUBLES)()
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_stats_read(self._handle, _ptr(self.state), buf, _stream()))
        return dict(zip(N.STAT_NAMES_PERFORMANCE if self.tracks_performance else N.STAT_NAMES, list(buf)))

    def step_perf(self, region, n_regions, prev_cells, next_cells, perf):
        self._check(region, torch.uint8, (self.cells,), "region")
        self._check(prev_cells, torch.int32, (self.num_envs,), "prev_cells")
        self._check(next_cells, torch.int32, (self.num_envs,), "next_cells")
        self._check(perf, torch.float32, (self.num_envs,), "perf")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_step_perf(_ptr(region), self.cells, int(n_regions), _ptr(prev_cells),
                                           _ptr(next_cells), self.num_envs, _ptr(perf), _stream()))

    def discounted_returns(self, reward, flags, gamma, discount=None, bootstrap=None, out=None):
        """[T, n] rewards/flags -> [T, n] discounted returns on the device (actor_critic.py:115-135)."""
        T = reward.shape[0]
        n = self.num_envs
        self._check(reward, torch.float32, (T, n), "reward")
        self._check(flags, torch.uint8, (T, n), "flags")
        if discount is not None:
            self._check(discount, torch.float32, (T, n), "discount")
        if bootstrap is not None:
            self._check(bootstrap, torch.float32, (n,), "bootstrap")
        if out is None:
            out = torch.empty_like(reward)
        self._check(out, torch.float32, (T, n), "returns")
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_discounted_returns(_ptr(reward), _ptr(discount), _ptr(flags), _ptr(bootstrap), T, n,
                                                    float(gamma), _ptr(out), _stream()))
        return out

    # -- helpers --------------------------------------------------------------------------------------------
    def _check(self, t, dtype, shape, what):
        if not isinstance(t, torch.Tensor):
            raise TypeError("%s must be a torch tensor" % what)
        if t.device != self.device:
            raise ValueError("%s must live on %s (got %s)" % (what, self.device, t.device))
        if t.dtype != dtype:
            raise ValueError("%s must have dtype %s (got %s)" % (what, dtype, t.dtype))
        if tuple(t.shape) != tuple(shape):
            raise ValueError("%s must have shape %s (got %s)" % (what, tuple(shape), tuple(t.shape)))
        if not t.is_contiguous():
            raise ValueError("%s must be contiguous" % what)
        return t


class BoardMapper(object):
    """Device value table + the `cx_board_mapper_apply` launch: boards -> arrays of mapped values.

    The device side of `rendering.ObservationToArray` / `ObservationToFeatureArray`
    (campx/rendering.py:461-712).  `values` is a numpy array `[256, depth]` (the value of every byte a
    board may hold), `known` a `[256]` bool array saying which bytes the mapping really covers.
    """

    def __init__(self, values, known, device=None):
        import numpy as np
        N.require_cuda()
        self._lib = N.load()
        values = np.ascontiguousarray(values)
        if values.ndim != 2 or values.shape[0] != 256:
            raise ValueError("values must have shape [256, depth]")
        known = np.ascontiguousarray(known, dtype=np.uint8)
        if known.shape != (256,):
            raise ValueError("known must have shape [256]")
        self.depth = int(values.shape[1])
        self.np_dtype = values.dtype
        self.elem_size = int(values.dtype.itemsize)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise N.NativeLibraryError("campx_b200 runs on CUDA devices only (got %s)" % self.device)
        self._handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_board_mapper_create(values.ctypes.data_as(ctypes.c_void_p),
                                                     known.ctypes.data_as(ctypes.c_void_p), self.depth,
                                                     self.elem_size, ctypes.byref(self._handle)))

    def close(self):
        if getattr(self, "_handle", None) is not None and self._handle.value:
            self._lib.cx_board_mapper_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def apply(self, board, out, permute=None, unknown=None):
        """board uint8 [..., rows, cols] (contiguous) -> out [n_boards * depth * rows * cols] elements, in the
        axis order `permute` asks for.  `unknown`: int32[1] device counter, nonzero afterwards if a board held
        a byte outside the mapping."""
        if board.dtype != torch.uint8 or not board.is_contiguous() or board.device != self.device:
            raise ValueError("board must be a contiguous uint8 tensor on %s" % self.device)
        rows, cols = int(board.shape[-2]), int(board.shape[-1])
        nb = board.numel() // (rows * cols)
        if out.device != self.device or not out.is_contiguous() or out.element_size() != self.elem_size \
                or out.numel() != nb * self.depth * rows * cols:
            raise ValueError("out must be a contiguous tensor of %d %d-byte elements on %s"
                             % (nb * self.depth * rows * cols, self.elem_size, self.device))
        perm = None if permute is None else (ctypes.c_int32 * 3)(*[int(p) for p in permute])
        with torch.cuda.device(self.device):
            N.check(self._lib.cx_board_mapper_apply(self._handle, _ptr(board), nb, rows, cols, perm, _ptr(out),
                                                    _ptr(unknown), _stream()))
        return out
