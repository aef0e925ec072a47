"""cx_policy_sample_board: the reference's acting policy (examples/actor_critic.py:64-98) evaluated on the layered board
read off the uint8 board, for every occluded world -- single-agent and generic, of any board size -- with the bits of
cx_policy_sample on the expanded float32 planes wherever that kernel takes the input."""
import numpy as np
import pytest
import torch

from campx_b200 import things
from campx_b200 import _native as N
from campx_b200.ascii_art import Partial, ascii_art_to_game
from examples.actor_critic_batched import GraphedRollout, Policy, needs_board_policy, run_graphed
from examples.worlds import Walker, make_world
from oracle import campx_oracle as O

pytestmark = pytest.mark.gpu


def _random_world(rows, cols, seed, n, **kw):
    rng = np.random.Generator(np.random.PCG64(seed))
    cells = rng.random((rows, cols))
    art = np.full((rows, cols), ' ', dtype='<U1')
    art[cells < 0.25] = '#'
    art[(cells >= 0.25) & (cells < 0.45)] = '*'
    art[int(rng.integers(0, rows)), int(rng.integers(0, cols))] = 'A'
    art = [''.join(row) for row in art]
    return ascii_art_to_game(art, ' ', drapes={'A': Partial(Walker, walls='#', treasures='*'),
                                               '#': things.FixedDrape, '*': things.FixedDrape},
                             z_order='*A#', num_envs=n, **kw)


def _sprite_only_world(n):
    class Slider(things.Sprite):
        def update(self, actions, board, layers, backdrop, all_things, the_plot):
            if actions is None or actions > 3:
                return
            d = [(0, -1), (0, 1), (-1, 0), (1, 0)][actions]
            self._position = self.Position((self.position.row + d[0]) % self.corner.row,
                                           (self.position.col + d[1]) % self.corner.col)

    return ascii_art_to_game(['P..x', '....', 'Q...'], '.', sprites={'P': Slider, 'Q': Slider}, num_envs=n)


def _mid_rollout_board(game, steps=13, seed=5):
    game.its_showtime()
    boards = game.rollout(game.native.fill_actions(steps, seed=seed))[0]
    return boards[-1].contiguous()


def _weights(nat, n_hidden, seed):
    torch.manual_seed(seed)
    pol = Policy(nat.n_chars * nat.cells, n_hidden=n_hidden, n_actions=nat.n_actions).cuda()
    w = (pol.affine1.weight.detach().t().contiguous(), pol.affine1.bias.detach(), pol.action_head.weight.detach(),
         pol.action_head.bias.detach())
    return pol, w


def _planes(nat, board):
    return nat.layers_from_board(board, dtype=torch.float32).view(board.shape[0], -1)


def _outputs(nat, n):
    return (torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.float32, device="cuda"),
            torch.empty((n, nat.n_actions), dtype=torch.float32, device="cuda"))


@pytest.mark.parametrize("case", ["boat_race", "demo3", "random_8x12", "sprite_only"])
def test_bits_equal_policy_sample_on_the_planes(case):
    """Actions, log-probs and logits are torch.equal to cx_policy_sample on cx_layers_from_board_f32 of the same boards
    (boards taken mid-rollout after random actions; same seed, step and step_offset)."""
    n, n_hidden = {"boat_race": (4096, 32), "demo3": (333, 17), "random_8x12": (256, 32), "sprite_only": (100, 32)}[case]
    if case == "random_8x12":
        game = _random_world(8, 12, 4, n)
    elif case == "sprite_only":
        game = _sprite_only_world(n)
    else:
        game = make_world(case, num_envs=n, max_episode_steps=9)
    board = _mid_rollout_board(game)
    nat = game.native
    _, (w1t, b1, w2, b2) = _weights(nat, n_hidden, 1)
    step = torch.full((1,), 7, dtype=torch.int64, device="cuda")
    a1, l1, g1 = _outputs(nat, n)
    a2, l2, g2 = _outputs(nat, n)
    nat.policy_sample_board(board, w1t, b1, w2, b2, 11, step=step, step_offset=3, out=a1, logp=l1, logits_out=g1)
    nat.policy_sample(_planes(nat, board), w1t, b1, w2, b2, 11, step=step, step_offset=3, out=a2, logp=l2, logits_out=g2)
    assert torch.equal(g1, g2) and torch.equal(a1, a2) and torch.equal(l1, l2)
    assert len(torch.unique(a1)) > 1
    if case == "sprite_only":
        # the zeroed canvas: bytes that are no character set no input
        assert bool((board == 0).any())
        assert int(_planes(nat, board).sum()) == int((board != 0).sum())


@pytest.mark.parametrize("n,n_hidden", [(4096, 32), (77, 32), (77, 17)])
def test_hello_world_samples_on_the_device(n, n_hidden):
    """Hello World (7 x 13 x 36 = 3,276 inputs: more than cx_policy_sample takes; a generic-kernel game): the logits
    are the torch module's on the expanded planes to rounding, actions and log-probs are what cx_sample_actions draws
    from those logits."""
    game = make_world("hello", num_envs=n, max_episode_steps=50)
    board = _mid_rollout_board(game)
    nat = game.native
    assert nat.n_chars * nat.cells == 3276 and needs_board_policy(nat)
    pol, (w1t, b1, w2, b2) = _weights(nat, n_hidden, 2)
    with torch.no_grad():
        pol.affine1.weight.mul_(8.0)                           # logits far enough apart to draw several actions
        w1t = pol.affine1.weight.t().contiguous()
    with pytest.raises(NotImplementedError):
        nat.policy_sample(_planes(nat, board), w1t, b1, w2, b2, 1)
    acts, logp, logits = _outputs(nat, n)
    step = torch.full((1,), 3, dtype=torch.int64, device="cuda")
    nat.policy_sample_board(board, w1t, b1, w2, b2, 9, step=step, step_offset=1, out=acts, logp=logp, logits_out=logits)
    with torch.no_grad():
        want = pol.action_logits(_planes(nat, board))
    assert torch.allclose(logits, want, rtol=1e-4, atol=1e-5), float((logits - want).abs().max())
    logp2 = torch.empty_like(logp)
    acts2 = nat.sample_actions(logits, 9, step=step, step_offset=1, logits=True, logp=logp2)
    assert torch.equal(acts, acts2) and torch.equal(logp, logp2)
    assert int(acts.max()) < nat.n_actions and len(torch.unique(acts)) > 1


def test_step_counter_under_a_cuda_graph():
    """A captured call reads the step counter on the device: equal steps draw equal actions, step + 1 fresh ones."""
    n = 4096
    game = make_world("hello", num_envs=n, max_episode_steps=50)
    board = _mid_rollout_board(game)
    nat = game.native
    _, (w1t, b1, w2, b2) = _weights(nat, 32, 3)
    step = torch.zeros(1, dtype=torch.int64, device="cuda")
    acts = torch.empty(n, dtype=torch.uint8, device="cuda")
    call = lambda: nat.policy_sample_board(board, w1t, b1, w2, b2, 5, step=step, out=acts)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call()
    graph.replay()
    first = acts.clone()
    graph.replay()
    assert torch.equal(acts, first)
    step += 1
    graph.replay()
    assert not torch.equal(acts, first)


@pytest.mark.parametrize("world", ["boat_race", "hello"])
def test_env_offset_draws_the_slice_of_the_full_batch(world):
    """A 333-env game fed envs k .. k+332 of a 4,096-env batch with env_offset=k draws exactly their actions."""
    big = make_world(world, num_envs=4096, max_episode_steps=40)
    board = _mid_rollout_board(big)
    small = make_world(world, num_envs=333, max_episode_steps=40)
    small.its_showtime()
    nb, ns = big.native, small.native
    _, (w1t, b1, w2, b2) = _weights(nb, 32, 4)
    a1, l1, g1 = _outputs(nb, 4096)
    nb.policy_sample_board(board, w1t, b1, w2, b2, 21, step_offset=2, out=a1, logp=l1, logits_out=g1)
    k = 1001
    a2, l2, g2 = _outputs(ns, 333)
    ns.policy_sample_board(board[k:k + 333], w1t, b1, w2, b2, 21, step_offset=2, env_offset=k, out=a2, logp=l2,
                           logits_out=g2)
    assert torch.equal(a2, a1[k:k + 333]) and torch.equal(l2, l1[k:k + 333]) and torch.equal(g2, g1[k:k + 333])


def test_two_launch_rollout_on_hello_world():
    """policy_sample_board + step, T times, captured in a CUDA graph: the recorded actions replayed through a fresh
    engine give the same boards, rewards and flags, and three envs obey the oracle step by step."""
    n, T, limit = 256, 30, 11
    game = make_world("hello", num_envs=n, max_episode_steps=limit, track_returns=True)
    game.its_showtime()
    nat = game.native
    torch.manual_seed(6)
    pol = Policy(nat.n_chars * nat.cells, n_actions=nat.n_actions).cuda()
    roll = GraphedRollout(game, pol, T).capture()
    assert roll.board_policy and roll.kernels_per_step == 2
    boards, actions, rewards, flags = roll.run()
    boards = roll._states
    assert len(torch.unique(actions)) > 1
    fresh = make_world("hello", num_envs=n, max_episode_steps=limit, track_returns=True)
    first = fresh.its_showtime()[0].board
    assert torch.equal(boards[0], first)
    b2, r2, _, f2 = fresh.rollout(actions.clone())
    assert torch.equal(boards[1:], b2) and torch.equal(rewards, r2) and torch.equal(flags, f2)
    assert bool(((flags & N.CX_FLAG_TRUNCATED) != 0).any())
    an, bn, rn, fn = actions.cpu().numpy(), boards.cpu().numpy(), rewards.cpu().numpy(), flags.cpu().numpy()
    for i in (0, n // 2, n - 1):
        for t, (o, rew, dsc, term, trunc, eng) in enumerate(
                O.rollout("hello", an[:, i], rebuild_on_done=True, max_episode_steps=limit)):
            assert np.array_equal(bn[t + 1, i], np.asarray(o.board).astype(np.uint8)), (i, t)
            assert (0.0 if rew is None else float(rew)) == float(rn[t, i]), (i, t)
            assert trunc == bool(fn[t, i] & N.CX_FLAG_TRUNCATED) and term == bool(fn[t, i] & N.CX_FLAG_TERMINATED)


def test_refusals():
    game = make_world("demo1", num_envs=64, occlusion_in_layers=False)
    board = _mid_rollout_board(game)
    nat = game.native
    _, (w1t, b1, w2, b2) = _weights(nat, 32, 7)
    with pytest.raises(NotImplementedError):
        nat.policy_sample_board(board, w1t, b1, w2, b2, 1)
    game = make_world("demo1", num_envs=64)
    board = _mid_rollout_board(game)
    nat = game.native
    _, (w1t, b1, w2, b2) = _weights(nat, 64, 7)
    with pytest.raises(ValueError):
        nat.policy_sample_board(board, w1t, b1, w2, b2, 1)
    _, (w1t, b1, w2, b2) = _weights(nat, 32, 7)
    nat.policy_sample_board(board, w1t, b1, w2, b2, 1)
    for bad_board in (board[:32], board.float(), board.view(64, -1)):
        with pytest.raises(ValueError):
            nat.policy_sample_board(bad_board, w1t, b1, w2, b2, 1)
    with pytest.raises(ValueError):
        nat.policy_sample_board(board, w1t[1:].contiguous(), b1, w2, b2, 1)


def test_actor_critic_example_on_hello_world():
    history, game, roll = run_graphed(world="hello", num_envs=512, steps=20, iterations=2, log=lambda *_: None)
    assert roll.board_policy and roll.graph is not None
    assert len(history) == 2 and all(np.isfinite(h[0]) for h in history)
    assert game.episode_stats()["env_steps"] == 2 * 20 * 512


def test_large_board_takes_the_dense_walk():
    """A 40 x 40 board (1,600 cells, 6,400 inputs): the per-env lists of set inputs do not fit shared memory, so every
    input is walked; the logits are the torch module's to rounding and the draw is cx_sample_actions' on them."""
    n = 200
    game = _random_world(40, 40, 12, n, max_episode_steps=30)
    board = _mid_rollout_board(game)
    nat = game.native
    assert nat.cells == 1600
    for n_hidden in (32, 17):
        pol, (w1t, b1, w2, b2) = _weights(nat, n_hidden, 8)
        with torch.no_grad():
            pol.affine1.weight.mul_(8.0)
            w1t = pol.affine1.weight.t().contiguous()
        acts, logp, logits = _outputs(nat, n)
        nat.policy_sample_board(board, w1t, b1, w2, b2, 13, step_offset=4, out=acts, logp=logp, logits_out=logits)
        with torch.no_grad():
            want = pol.action_logits(_planes(nat, board))
        assert torch.allclose(logits, want, rtol=1e-4, atol=1e-5), float((logits - want).abs().max())
        logp2 = torch.empty_like(logp)
        acts2 = nat.sample_actions(logits, 13, step_offset=4, logits=True, logp=logp2)
        assert torch.equal(acts, acts2) and torch.equal(logp, logp2) and len(torch.unique(acts)) > 1
