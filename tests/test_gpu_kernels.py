"""GPU parity of the kernels (through the C ABI) against the golden fixtures and the numpy oracle,
driving the native library with the hand-written primitive descriptions of tests/expected_specs.py."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import campx_oracle as O
from tests.expected_specs import expected_spec

pytestmark = pytest.mark.gpu

WORLDS = ["boat_race", "demo1", "demo2", "demo3", "demo4", "hello"]


@pytest.fixture(autouse=True, params=["auto", "wt64", "wt128", "wt256", "stg"])
def agent_kernel(request, monkeypatch):
    """Single-agent worlds run on several kernels: tiny batches take the lane-per-env kernels (cx_rollout's default),
    larger ones k_agent_rollout in one of three builds (64 / 128 / 256 envs per warp; 64 is what large multi-step
    rollouts take), single steps the stateless composer.  Every test of this module runs on all of them:
    CX_ROUTE=tile64 / tile128 / tile256 sends small batches to k_agent_rollout as well, in that build; "stg"
    (CX_ROUTE=lane) sends every batch of whole warps to the small-batch kernel (k_agent_rollout_lane: lane = env,
    STG.128 tile copies)."""
    if request.param == "stg":
        monkeypatch.setenv("CX_ROUTE", "lane")
    elif request.param != "auto":
        monkeypatch.setenv("CX_ROUTE", "tile" + request.param[2:])
    return request.param


def _game(world, n, **kw):
    from campx_b200.runtime import NativeGame
    return NativeGame(expected_spec(world, **kw), n)


def board_str(b):
    return "".join(chr(int(v)) for v in b.reshape(-1).tolist())


@pytest.mark.parametrize("world", WORLDS)
def test_golden_episodes_step_by_step(golden_dir, world):
    """Every golden episode, one env per episode, one cx_step per action."""
    from campx_b200 import _native as N
    with open(os.path.join(golden_dir, world + ".json")) as f:
        fx = json.load(f)
    eps = fx["episodes"]
    n = len(eps)
    g = _game(world, n, auto_reset=False)
    board, reward, flags, disc = g.alloc_outputs(discount=True)
    first = g.render().cpu()
    for i, ep in enumerate(eps):
        assert board_str(first[i]) == ep["frames"][0]["board"]
    T = max(len(ep["actions"]) for ep in eps)
    for t in range(T):
        acts = torch.tensor([ep["actions"][t] if t < len(ep["actions"]) else 4 for ep in eps], dtype=torch.uint8)
        g.step(acts.cuda(), board, reward, flags, disc)
        b, r, f, d = board.cpu(), reward.cpu(), flags.cpu(), disc.cpu()
        lay = g.layers_from_board(board).cpu()
        for i, ep in enumerate(eps):
            if t >= len(ep["actions"]):
                continue
            want = ep["frames"][t + 1]
            ctx = "%s/%s t=%d" % (world, ep["name"], t)
            assert board_str(b[i]) == want["board"], ctx
            assert (want["reward"] is None) == bool(f[i] & N.CX_FLAG_REWARD_NONE), ctx
            if want["reward"] is not None:
                assert float(r[i]) == want["reward"], ctx
            assert float(d[i]) == want["discount"], ctx
            assert bool(f[i] & N.CX_FLAG_TERMINATED) == (want["discount"] == 0.0), ctx
            for k, ch in enumerate(g.spec.chars):
                got = "".join(str(int(v)) for v in lay[i, k].reshape(-1).tolist())
                assert got == want["layers"][ch], ctx + " layer %r" % ch


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("n", [1, 5, 64, 272])
def test_random_rollout_vs_oracle(world, n):
    """Fused rollout with time limit + auto reset vs the oracle rebuilt at every episode end."""
    from campx_b200 import _native as N
    T, limit = 60, 25
    g = _game(world, n, max_episode_steps=limit, auto_reset=True, track_returns=True)
    rng = np.random.Generator(np.random.PCG64(7 + n))
    hi = 5
    acts = rng.integers(0, hi, size=(T, n)).astype(np.uint8)
    if world == "hello":  # make "quit" rarer so that episodes have some length
        acts[(acts == 4) & (rng.random((T, n)) < 0.8)] = 0
    board, reward, flags, disc = g.alloc_outputs(T, discount=True)
    g.rollout(torch.from_numpy(acts).cuda(), board, reward, flags, disc)
    b, r, f, d = board.cpu().numpy(), reward.cpu().numpy(), flags.cpu().numpy(), disc.cpu().numpy()
    check_envs = range(n) if n <= 64 else list(range(0, n, 17)) + [n - 1]
    episodes = 0
    for i in check_envs:
        for t, (obs, rew, dsc, term, trunc, eng) in enumerate(
                O.rollout(world, acts[:, i], rebuild_on_done=True, max_episode_steps=limit)):
            ctx = "%s env %d t %d" % (world, i, t)
            assert np.array_equal(b[t, i].reshape(-1), np.asarray(obs.board).reshape(-1).astype(np.uint8)), ctx
            assert (rew is None) == bool(f[t, i] & N.CX_FLAG_REWARD_NONE), ctx
            if rew is not None:
                assert float(rew) == float(r[t, i]), ctx
            assert float(dsc) == float(d[t, i]), ctx
            assert term == bool(f[t, i] & N.CX_FLAG_TERMINATED), ctx
            assert trunc == bool(f[t, i] & N.CX_FLAG_TRUNCATED), ctx
            episodes += term or trunc
    assert episodes > 0
    # step-by-step cx_step calls give the same thing as the fused rollout
    g2 = _game(world, n, max_episode_steps=limit, auto_reset=True, track_returns=True)
    b1, r1, f1, d1 = g2.alloc_outputs(discount=True)
    dacts = torch.from_numpy(acts).cuda()
    for t in range(T):
        g2.step(dacts[t].contiguous(), b1, r1, f1, d1)
        assert torch.equal(b1, board[t]) and torch.equal(r1, reward[t]) and torch.equal(f1, flags[t])
        assert torch.equal(d1, disc[t])
    g.fold_stats(), g2.fold_stats()   # the partial statistics blocks depend on the launch geometry
    if not torch.equal(g.state, g2.state):
        bad = (g.state != g2.state).nonzero().flatten().cpu().tolist()
        raise AssertionError("state blobs differ at byte offsets %s: %s vs %s; stats %s vs %s" % (
            bad[:16], g.state.cpu()[bad[:16]].tolist(), g2.state.cpu()[bad[:16]].tolist(), g.stats(), g2.stats()))
    # episode statistics agree with a host-side recomputation from the outputs
    done = (f & (N.CX_FLAG_TERMINATED | N.CX_FLAG_TRUNCATED)) != 0
    st = g.stats()
    assert st["episodes"] == done.sum()
    assert st["env_steps"] == T * n
    ret = np.zeros(n, np.float64)
    total = 0.0
    for t in range(T):
        ret += r[t]
        total += ret[done[t]].sum()
        ret[done[t]] = 0
    assert abs(st["return_sum"] - total) < 1e-6


@pytest.mark.parametrize("world", ["boat_race", "demo3"])
@pytest.mark.parametrize("n", [48, 1040, 1000])
def test_ragged_batches_run_their_aligned_part_on_the_vector_path(world, n):
    """A batch that is not a whole number of warp tiles: its aligned part takes the vector kernels (whole warps of
    k_agent_rollout_lane / whole tiles of k_agent_rollout), the rest one warp of the scalar path -- two launches that
    must give what one would (n % 16 == 0; n = 1000 has unaligned rows and runs on the scalar path altogether)."""
    from campx_b200 import _native as N
    T, limit = 40, 13
    g = _game(world, n, max_episode_steps=limit, auto_reset=True, track_returns=True)
    acts = g.fill_actions(T, seed=99)
    board, reward, flags, disc = g.alloc_outputs(T, discount=True)
    g.rollout(acts, board, reward, flags, disc)
    a, b, r, f = acts.cpu().numpy(), board.cpu().numpy(), reward.cpu().numpy(), flags.cpu().numpy()
    for i in sorted({0, 31, 32, n // 2, n - 17, n - 16, n - 1}):
        for t, (obs, rew, dsc, term, trunc, eng) in enumerate(
                O.rollout(world, a[:, i], rebuild_on_done=True, max_episode_steps=limit)):
            ctx = "%s env %d t %d" % (world, i, t)
            assert np.array_equal(b[t, i].reshape(-1), np.asarray(obs.board).reshape(-1).astype(np.uint8)), ctx
            assert (0.0 if rew is None else float(rew)) == float(r[t, i]), ctx
            assert term == bool(f[t, i] & N.CX_FLAG_TERMINATED) and trunc == bool(f[t, i] & N.CX_FLAG_TRUNCATED), ctx
    g2 = _game(world, n, max_episode_steps=limit, auto_reset=True, track_returns=True)
    b1, r1, f1, d1 = g2.alloc_outputs(discount=True)
    for t in range(T):
        g2.step(acts[t].contiguous(), b1, r1, f1, d1)
        assert torch.equal(b1, board[t]) and torch.equal(r1, reward[t]) and torch.equal(f1, flags[t])
    g.fold_stats(), g2.fold_stats()
    assert torch.equal(g.state, g2.state)
    assert g.stats()["env_steps"] == T * n
