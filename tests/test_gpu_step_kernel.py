"""GPU parity of the single-step composer (`k_agent_step_flat`: cx_step / cx_step_observations on single-agent
games) and of `cx_sample_actions`.

The composer must agree with (a) the tile kernels it replaces for T = 1 (`CX_ROUTE=no_step_composer` routes single
steps through them again), (b) `cx_layers_from_board[_f32]` on the board it wrote, for every element type, ragged batch
sizes included, and (c) the CPU oracle.  The reference encoding of the float planes is
`board.layered_board.view(-1).float()` (examples/actor_critic.py:147,173)."""
import numpy as np
import pytest
import torch

from campx_b200 import _native as N
from examples.worlds import make_world
from oracle import campx_oracle as O
from tests.expected_specs import expected_spec

pytestmark = pytest.mark.gpu

AGENT_WORLDS = ["boat_race", "demo1", "demo2", "demo3", "demo4"]


def _game(world, n, **kw):
    from campx_b200.runtime import NativeGame
    return NativeGame(expected_spec(world, **kw), n)


@pytest.mark.parametrize("world", AGENT_WORLDS)
@pytest.mark.parametrize("n,kw", [
    (1, dict()),
    (5, dict(max_episode_steps=7, track_returns=True)),
    (64, dict(max_episode_steps=9, auto_reset=False)),                 # frozen envs after the limit
    (272, dict(max_episode_steps=11, track_returns=True)),
    (4096 + 7, dict(max_episode_steps=10, track_returns=True)),        # ragged tail in the last CTA
])
def test_single_step_composer_equals_tile_kernels(world, n, kw, monkeypatch):
    """T = 1 through the composer == T = 1 through the tile kernels: outputs and the whole state blob."""
    T = 26
    a, b = _game(world, n, **kw), _game(world, n, **kw)
    acts = a.fill_actions(T, seed=5)
    acts[3, ::7] = 9                                                    # a few actions outside the action set
    oa, ob = a.alloc_outputs(discount=True), b.alloc_outputs(discount=True)
    for t in range(T):
        monkeypatch.delenv("CX_ROUTE", raising=False)
        a.step(acts[t].contiguous(), *oa)
        monkeypatch.setenv("CX_ROUTE", "no_step_composer")
        b.step(acts[t].contiguous(), *ob)
        for x, y, what in zip(oa, ob, ("board", "reward", "flags", "discount")):
            assert torch.equal(x, y), (world, n, t, what)
    a.fold_stats(), b.fold_stats()
    assert torch.equal(a.state, b.state)
    assert a.stats() == b.stats()


def test_unknown_route_fails_the_call(monkeypatch):
    """CX_ROUTE names one kernel route; a name it does not know fails the call instead of running the automatic
    choice."""
    g = _game("boat_race", 64)
    acts = g.fill_actions(4, seed=1)
    monkeypatch.setenv("CX_ROUTE", "tile32")
    with pytest.raises(ValueError, match="unknown CX_ROUTE 'tile32'"):
        g.step(acts[0].contiguous(), *g.alloc_outputs())
    with pytest.raises(ValueError, match="unknown CX_ROUTE 'tile32'"):
        g.rollout(acts, *g.alloc_outputs(4))


@pytest.mark.parametrize("world", AGENT_WORLDS)
@pytest.mark.parametrize("dtype", [torch.uint8, torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n", [1, 50, 77, 1024, 65536])
def test_step_observations_planes_equal_layers_of_the_board(world, dtype, n):
    """Board and typed planes from ONE launch; planes == (board == chars[k]) in canonical channel order, as 0 / 1."""
    T = 12
    g = _game(world, n, max_episode_steps=5, track_returns=True)
    h = _game(world, n, max_episode_steps=5, track_returns=True)
    acts = g.fill_actions(T, seed=9)
    board, reward, flags, _ = g.alloc_outputs()
    planes = torch.empty((n, g.n_chars, g.rows, g.cols), dtype=dtype, device="cuda")
    b2, r2, f2, _ = h.alloc_outputs()
    for t in range(T):
        planes.fill_(7)                                                 # every element must be overwritten
        g.step_observations(acts[t].contiguous(), board, planes, reward, flags)
        h.step(acts[t].contiguous(), b2, r2, f2)
        assert torch.equal(board, b2) and torch.equal(reward, r2) and torch.equal(flags, f2)
        want = h.layers_from_board(b2)                                  # uint8, derived from the finished board
        assert torch.equal(planes, want.to(dtype)), (world, dtype, n, t)
    g.fold_stats(), h.fold_stats()
    assert torch.equal(g.state, h.state)


def test_step_observations_against_the_oracle():
    """float32 planes, reward, flags of cx_step_observations == the CPU oracle's layered_board.float() et al."""
    n, T, limit = 96, 40, 13
    g = _game("boat_race", n, max_episode_steps=limit, track_returns=True)
    acts = g.fill_actions(T, seed=3)
    board, reward, flags, _ = g.alloc_outputs()
    planes = torch.empty((T, n, g.n_chars, g.rows, g.cols), dtype=torch.float32, device="cuda")
    rs, fs = [], []
    for t in range(T):
        g.step_observations(acts[t].contiguous(), board, planes[t], reward, flags)
        rs.append(reward.clone())
        fs.append(flags.clone())
    a, p = acts.cpu().numpy(), planes.cpu().numpy()
    r, f = torch.stack(rs).cpu().numpy(), torch.stack(fs).cpu().numpy()
    for i in (0, 31, 32, n - 1):
        for t, (o, rew, dsc, term, trunc, eng) in enumerate(
                O.rollout("boat_race", a[:, i], rebuild_on_done=True, max_episode_steps=limit)):
            assert np.array_equal(p[t, i], np.asarray(o.layered_board).astype(np.float32)), (i, t)
            assert float(rew) == float(r[t, i]) and trunc == bool(f[t, i] & N.CX_FLAG_TRUNCATED), (i, t)


def test_step_observations_on_a_generic_game_takes_the_two_kernel_route():
    n = 48
    g = _game("hello", n, max_episode_steps=6)
    h = _game("hello", n, max_episode_steps=6)
    acts = g.fill_actions(8, seed=1)
    board, reward, flags, disc = g.alloc_outputs()
    b2, r2, f2, d2 = h.alloc_outputs()
    for dtype in (torch.uint8, torch.float32):
        planes = torch.empty((n, g.n_chars, g.rows, g.cols), dtype=dtype, device="cuda")
        for t in range(4):
            g.step_observations(acts[t].contiguous(), board, planes, reward, flags, disc)
            h.step(acts[t].contiguous(), b2, r2, f2, d2)
            assert torch.equal(board, b2) and torch.equal(planes, h.layers_from_board(b2).to(dtype))
    with pytest.raises(NotImplementedError):
        g.step_observations(acts[0].contiguous(), board,
                            torch.empty((n, g.n_chars, g.rows, g.cols), dtype=torch.bfloat16, device="cuda"),
                            reward, flags, disc)


def test_engine_play_emits_the_planes_the_caller_reads():
    """A caller that read float32 planes of the last Observation gets the next ones from the step kernel itself
    (no second launch); values equal the lazily derived ones."""
    n = 1000
    a = make_world("boat_race", num_envs=n, max_episode_steps=10)
    b = make_world("boat_race", num_envs=n, max_episode_steps=10)
    oa, _, _ = a.its_showtime()
    ob, _, _ = b.its_showtime()
    b.fused_observation_steps = False
    acts = a.native.fill_actions(15, seed=2)
    for t in range(15):
        pa = oa.layered_board_as(torch.float32)
        pb = ob.layered_board_as(torch.float32)
        assert torch.equal(pa, pb) and pa.dtype == torch.float32
        oa, ra, _ = a.play(acts[t])
        ob, rb, _ = b.play(acts[t])
        assert torch.float32 in oa._planes and torch.float32 not in ob._planes     # pre-filled vs lazy
        assert torch.equal(oa.board, ob.board) and torch.equal(ra, rb)
    assert torch.equal(oa.layered_board, ob.layered_board)


def test_step_counter_saturates_instead_of_freezing_the_env():
    """ADVICE r1: the 15-bit per-env step counter shares its word with the OVER bit.  An episode without a time
    limit that runs past 32,767 steps must keep stepping (it used to set the OVER bit by itself and freeze)."""
    n, T = 64, 4096
    g = _game("boat_race", n, max_episode_steps=0, track_returns=True, auto_reset=True)
    board, reward, flags, _ = g.alloc_outputs(T)
    for i in range(9):                                                  # 36,864 steps
        g.rollout(g.fill_actions(T, seed=4, t0=i * T), board, reward, flags)
    assert int((flags & N.CX_FLAG_ALREADY_OVER).max()) == 0
    assert float(reward.min()) <= -1.0 and float(reward.max()) >= 0.0  # still paying the per-step toll / bonuses
    steps, _ = g.episode_state()
    assert int(steps.min()) == 0x7FFF and int(steps.max()) == 0x7FFF
    b1, r1, f1, _ = g.alloc_outputs()
    g.step(g.fill_actions(1, seed=8)[0].contiguous(), b1, r1, f1)       # the single-step kernel agrees
    assert int((f1 & N.CX_FLAG_ALREADY_OVER).max()) == 0
    assert g.stats()["env_steps"] == n * (9 * T + 1)


def test_sample_actions_is_the_categorical_distribution():
    n, A = 1 << 18, 5
    g = _game("boat_race", n)
    probs = torch.tensor([0.1, 0.0, 0.45, 0.25, 0.2], device="cuda").repeat(n, 1).contiguous()
    step = torch.zeros(1, dtype=torch.int64, device="cuda")
    a0 = g.sample_actions(probs, seed=11, step=step)
    assert a0.dtype == torch.uint8 and int(a0.max()) < A
    freq = torch.bincount(a0.long(), minlength=A).double() / n
    assert float(freq[1]) == 0.0                                        # a zero-probability action is never drawn
    assert float((freq - probs[0].double()).abs().max()) < 0.005        # ~5 sigma at n = 2^18
    assert torch.equal(a0, g.sample_actions(probs, seed=11, step=step))               # counter-based: reproducible
    assert not torch.equal(a0, g.sample_actions(probs, seed=11, step=step, step_offset=1))
    step += 1                                                           # ... and a device-side counter advances it
    assert torch.equal(g.sample_actions(probs, seed=11, step=step),
                       g.sample_actions(probs, seed=11, step=None, step_offset=1))
    # logits: softmax inside the kernel == probabilities handed in; log-probabilities come out on request
    logits = torch.randn(n, A, device="cuda")
    logp = torch.empty(n, device="cuda")
    al = g.sample_actions(logits, seed=3, logits=True, logp=logp)
    sm = torch.softmax(logits, dim=1)
    ap = g.sample_actions(sm.contiguous(), seed=3)
    assert float((al != ap).double().mean()) < 1e-4                     # identical up to rounding at bin edges
    want = torch.log_softmax(logits, dim=1).gather(1, al.long().view(-1, 1)).squeeze(1)
    assert float((logp - want).abs().max()) < 1e-4
    # independent envs: neighbouring envs do not share draws
    assert float((a0[::2] == a0[1::2]).double().mean()) < 0.5
