#!/usr/bin/env python
"""Actor-critic on boat_race with the whole rollout on the GPU (BASELINE config 5).

The reference's examples/actor_critic.py steps ONE environment on the CPU, builds a fresh game per
episode and runs its policy once per step.  Here 4,096 environments step together:

  state   = layered_board as float32 [N, 7*5*5=175]  (actor_critic.py:147,173 `layered_board.view(-1).float()`)
            written by the step kernel itself (cx_step_observations), next to the board
  policy  = Linear(175,32) -> ReLU -> {Linear(32,5) softmax, Linear(32,1)}   (actor_critic.py:64-86)
  action  ~ Categorical(probs)                                                (actor_critic.py:90-98)
  step    = Engine.play(action indices)            one cx_step launch, time limit 100 + auto reset
  returns = cx_discounted_returns over the [T, N] rewards on the device       (actor_critic.py:115-122)
  loss    = -(log pi) * (R - V) + smooth_l1(V, R), Adam                        (actor_critic.py:123-135)

Other worlds (--world hello, ...): where the policy input is larger than cx_policy_sample takes, or the game runs on
the generic kernels, the rollout stores the uint8 boards instead of float32 planes and the policy reads them directly
(cx_policy_sample_board); the learner's affine1 is an embedding_bag over the set inputs of each board.

Nothing leaves the device inside an iteration.  The network itself is ordinary torch and is not part of
the hand-written hot path; the environment, observation encoding and return scan are.
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch
import torch.nn as nn
import torch.nn.functional as F

from campx_b200 import _native as N
from examples.worlds import BOAT_RACE_REGIONS, make_world


class Policy(nn.Module):
    def __init__(self, n_inputs=175, n_hidden=32, n_actions=5):
        super().__init__()
        self.affine1 = nn.Linear(n_inputs, n_hidden)
        self.action_head = nn.Linear(n_hidden, n_actions)
        self.value_head = nn.Linear(n_hidden, 1)

    def forward(self, x):
        x = F.relu(self.affine1(x))
        return F.softmax(self.action_head(x), dim=-1), self.value_head(x).squeeze(-1)

    def action_logits(self, x):
        """The acting half only (no value head, no softmax): what a rollout step needs."""
        return self.action_head(F.relu(self.affine1(x)))

    def forward_indices(self, idx):
        """forward() on layered boards given by the indices of their set inputs (int [B, cells], board_indices):
        affine1 is the sum of the W1^T rows of those inputs plus the bias -- the same function as affine1 on the
        0/1 planes, differentiable in the weight, without the [B, n_inputs] float planes."""
        w1 = self.affine1.weight
        w1t = torch.cat([w1.t(), w1.new_zeros(1, w1.shape[0])])            # row n_inputs: "no character"
        h = F.embedding_bag(idx, w1t, mode="sum", padding_idx=w1.shape[1]) + self.affine1.bias
        x = F.relu(h)
        return F.softmax(self.action_head(x), dim=-1), self.value_head(x).squeeze(-1)


def board_indices(boards, chars, cells):
    """uint8 boards [..., rows, cols] -> int32 [..., cells]: the input index k * cells + cell of the one set input of every
    cell in the layered board (channel k = (board == chars[k]), rendering.py:204-215), or n_chars * cells where the
    byte is no character of the game."""
    n_chars = len(chars)
    lut = torch.full((256,), -1, dtype=torch.int32, device=boards.device)
    lut[torch.tensor([ord(c) for c in chars], dtype=torch.long, device=boards.device)] = torch.arange(
        n_chars, dtype=torch.int32, device=boards.device)
    k = lut[boards.reshape(boards.shape[:-2] + (cells,)).long()]
    cell = torch.arange(cells, dtype=torch.int32, device=boards.device)
    return torch.where(k >= 0, k * cells + cell, torch.full_like(k, n_chars * cells))


def needs_board_policy(nat):
    """True where cx_policy_sample cannot run the rollout on float32 planes: the game runs on the generic kernels, or
    cx_policy_sample refuses the input size (NotImplementedError: the limit is its launcher's, cx_aux_kernels.cu, and
    is asked rather than restated here -- one launch on zeros)."""
    if nat.info.path != N.CX_PATH_AGENT:
        return True
    feat, n, A = nat.n_chars * nat.cells, nat.num_envs, nat.n_actions
    zeros = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=nat.device)
    try:
        nat.policy_sample(zeros(n, feat), zeros(feat, 32), zeros(32), zeros(A, 32), zeros(A), 0)
    except NotImplementedError:
        return True
    return False


def world_kwargs(world):
    """boat_race also keeps its hidden safety performance (examples/boat_race.py:117-151) inside the step kernels: the
    reference's P (reinforce.py:186-194), logged next to the reward; so does sprite_race, boat_race with a sprite agent."""
    return {"performance_regions": BOAT_RACE_REGIONS} if world in ("boat_race", "sprite_race") else {}


def performance_note(nat, before):
    """" mean episode performance X" over the episodes finished since the stats() dict `before` ("" for worlds that do
    not track it); returns (note, stats now)"""
    now = nat.stats()
    if "performance_sum" not in now:
        return "", now
    episodes = now["episodes"] - before["episodes"]
    mean = (now["performance_sum"] - before["performance_sum"]) / episodes if episodes else float("nan")
    return "  mean episode performance %.2f" % mean, now


def run(num_envs=4096, steps=100, iterations=5, gamma=0.99, lr=3e-2, seed=543, log=print, device="cuda"):
    torch.manual_seed(seed)
    game = make_world("boat_race", num_envs=num_envs, max_episode_steps=steps, track_returns=True,
                      **world_kwargs("boat_race"))
    obs, _, _ = game.its_showtime()
    nat = game.native
    seen = nat.stats()
    policy = Policy().to(device)
    optimizer = torch.optim.Adam(policy.parameters(), lr=lr)
    eps = torch.finfo(torch.float32).eps
    history = []
    for it in range(iterations):
        t0 = time.time()
        log_probs, values, rewards, flags = [], [], [], []
        for _ in range(steps):
            state = obs.layered_board_as(torch.float32).view(num_envs, -1)      # [N, 175] on the device
            probs, value = policy(state)
            dist = torch.distributions.Categorical(probs)
            action = dist.sample()
            obs, reward, _ = game.play(action)
            log_probs.append(dist.log_prob(action))
            values.append(value)
            rewards.append(reward.clone())
            flags.append(game.flags.clone())
        rewards, flags = torch.stack(rewards), torch.stack(flags)
        returns = nat.discounted_returns(rewards, flags, gamma)                 # [T, N], device scan
        returns = (returns - returns.mean()) / (returns.std() + eps)
        log_probs, values = torch.stack(log_probs), torch.stack(values)
        advantage = returns - values.detach()
        loss = (-log_probs * advantage).mean() + F.smooth_l1_loss(values, returns)
        optimizer.zero_grad()
        loss.backward()
        optimizer.step()
        mean_reward = float(rewards.mean())
        dt = time.time() - t0
        history.append((float(loss.detach()), mean_reward))
        note, seen = performance_note(nat, seen)
        log("iter %d  loss %.4f  mean step reward %.4f%s  %.0f env-steps/s incl. policy fwd/bwd" % (
            it, float(loss.detach()), mean_reward, note, num_envs * steps / dt))
    return history, game


class GraphedRollout(object):
    """One T-step rollout (policy -> sample -> Engine.play, T times) captured ONCE as a CUDA graph and replayed
    per iteration.  A 4,096-env step is launch-bound on a B200 (it moves 3 MB), so the loop is built from as few
    launches as the reference's data flow allows -- two per env-batch step:

        cx_policy_sample                          the acting half of the policy in one kernel: Linear(175,32), ReLU,
                                                  Linear(32,5), softmax and Categorical.sample()
                                                  (actor_critic.py:64-98); weights are read from the torch module
        cx_step_observations                      Engine.play() that writes the NEXT policy input -- the layered
                                                  board as float32 planes (actor_critic.py:147,173) -- together with
                                                  board, reward and flags, straight into the rollout buffers

    (fused_policy=False keeps the policy in torch: Linear, ReLU, Linear, then cx_sample_actions -- five launches.)
    Games that need_board_policy() store boards [T + 1, N, rows, cols] uint8 instead of planes, two launches per step:

        cx_policy_sample_board                    the same policy read off the uint8 board of every env
        cx_step                                   Engine.play() writing the next board straight into the rollout buffer

    (with fused_policy=False: cx_layers_from_board_f32, the torch policy and cx_sample_actions.)
    persistent=True goes one step further: cx_rollout_policy runs the WHOLE T-step loop in one launch (a CTA owns 32 envs,
    their policy input stays in shared memory and changes by four floats per step); bit-identical to the two-launch loop.

    The rollout runs under no_grad into static buffers (states, actions, rewards, flags); the learner then
    re-evaluates the policy on all T*N states in one batched forward pass (the usual A2C/PPO split).
    """

    def __init__(self, game, policy, steps, seed=543, fused_policy=None, persistent=False):
        self.game, self.policy, self.T, self.seed = game, policy, int(steps), int(seed)
        if fused_policy is None:
            fused_policy = policy.affine1.out_features <= 32
        self.fused_policy = bool(fused_policy)
        nat = game.native
        self.board_policy = needs_board_policy(nat)
        self.persistent = bool(persistent) and self.fused_policy and game.num_envs % 32 == 0 and not self.board_policy
        n, dev = game.num_envs, nat.device
        self.feat = nat.n_chars * nat.cells
        if self.board_policy:
            self._states = torch.empty((self.T + 1, n, nat.rows, nat.cols), dtype=torch.uint8, device=dev)
        else:
            self._states = torch.empty((self.T + 1, n, self.feat), dtype=torch.float32, device=dev)
        self.actions = torch.empty((self.T, n), dtype=torch.uint8, device=dev)
        self.rewards = torch.empty((self.T, n), dtype=torch.float32, device=dev)
        self.flags = torch.empty((self.T, n), dtype=torch.uint8, device=dev)
        self.board = torch.empty((n, nat.rows, nat.cols), dtype=torch.uint8, device=dev)
        self.all_envs = torch.ones(n, dtype=torch.uint8, device=dev)
        self.step = torch.zeros(1, dtype=torch.int64, device=dev)      # Philox step counter, advanced inside the graph
        # every rollout starts from the its_showtime frame: its planes are the same for every env and rollout
        first = game.reset(self.all_envs)
        if self.board_policy:
            self._states[0].copy_(first.board)
        else:
            self._states[0].copy_(first.layered_board_as(torch.float32).view(n, -1))
        self.graph = None
        self.step_kernel = ("cx_policy_sample (k_policy_sample: policy MLP + softmax + sample) + " if self.fused_policy else "") + \
            "cx_step_observations (k_agent_step_flat: board + float32 planes + reward + flags)"
        self.kernels_per_step = 2 if self.fused_policy else 5
        if self.board_policy:
            self.step_kernel = ("cx_policy_sample_board (k_policy_sample_board: policy MLP on the uint8 board + softmax + "
                                "sample) + " if self.fused_policy else "") + "cx_step (board + reward + flags)"
            self.kernels_per_step = 2 if self.fused_policy else 4
        if self.persistent:
            self.step_kernel = "cx_rollout_policy (k_agent_policy_rollout: policy + sample + play + float32 planes, T steps per launch)"
            self.kernels_per_step = 1.0 / self.T
        self.w1t = torch.empty((self.feat, policy.affine1.out_features), dtype=torch.float32, device=dev)

    @property
    def states(self):
        """float32 [T, N, L*R*C] (uint8 boards [T, N, R, C] where board_policy): states[t] is what the policy saw
        before action t."""
        return self._states[:self.T]

    def _body(self):
        nat, game, n = self.game.native, self.game, self.game.num_envs
        with torch.no_grad():
            p = self.policy
            if self.fused_policy:                               # affine1.weight transposed, once per rollout
                self.w1t.copy_(p.affine1.weight.t())
            for t in range(0 if self.persistent else self.T):
                if self.board_policy:
                    if self.fused_policy:
                        nat.policy_sample_board(self._states[t], self.w1t, p.affine1.bias, p.action_head.weight,
                                                p.action_head.bias, self.seed, step=self.step, step_offset=t,
                                                out=self.actions[t])
                    else:
                        logits = p.action_logits(nat.layers_from_board(self._states[t], dtype=torch.float32).view(n, -1))
                        nat.sample_actions(logits, self.seed, step=self.step, step_offset=t, logits=True,
                                           out=self.actions[t])
                    nat.step(self.actions[t], self._states[t + 1], self.rewards[t], self.flags[t])
                    continue
                if self.fused_policy:
                    nat.policy_sample(self._states[t], self.w1t, p.affine1.bias, p.action_head.weight,
                                      p.action_head.bias, self.seed, step=self.step, step_offset=t, out=self.actions[t])
                else:
                    logits = p.action_logits(self._states[t])
                    nat.sample_actions(logits, self.seed, step=self.step, step_offset=t, logits=True, out=self.actions[t])
                nat.step_observations(self.actions[t], self.board, self._states[t + 1], self.rewards[t], self.flags[t])
            if self.persistent:
                nat.rollout_policy(self.T, self.w1t, p.affine1.bias, p.action_head.weight, p.action_head.bias, self.seed,
                                   self._states, self.actions, self.rewards, self.flags, step=self.step)
            self.step.add_(self.T)
            # a fresh episode for every env, like the reference's make_game() per episode (actor_critic.py:146):
            # a masked reset keeps the episode statistics
            nat.reset(self.all_envs)

    def capture(self):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                    # warm-up off the capture (lazy kernel configuration)
            self._body()
        torch.cuda.current_stream().wait_stream(side)
        if self.board_policy:
            # the warm-up is not part of the run: a full reset also zeroes the statistics, so that episode_stats()
            # counts the replayed iterations only.  The plane modes keep counting the warm-up rollout, as they always
            # have (a known difference between the modes: their statistics include one extra rollout).
            self.game.native.reset()
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._body()
        return self

    def run(self):
        if self.graph is None:
            self._body()
        else:
            self.graph.replay()
        return self.states, self.actions, self.rewards, self.flags


def run_graphed(num_envs=4096, steps=100, iterations=5, gamma=0.99, lr=3e-2, seed=543, log=print, device="cuda",
                use_graph=True, persistent=False, world="boat_race"):
    """Same learner as run(), rollout replayed from a CUDA graph.  Returns (history, game, rollout)."""
    torch.manual_seed(seed)
    game = make_world(world, num_envs=num_envs, max_episode_steps=steps, track_returns=True, **world_kwargs(world))
    game.its_showtime()
    nat = game.native
    policy = Policy(nat.n_chars * nat.cells, n_actions=nat.n_actions).to(device)
    optimizer = torch.optim.Adam(policy.parameters(), lr=lr)
    eps = torch.finfo(torch.float32).eps
    roll = GraphedRollout(game, policy, steps, persistent=persistent)
    if use_graph:
        roll.capture()
    history = []
    seen = nat.stats()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    for it in range(iterations):
        e0.record()
        states, actions, rewards, flags = roll.run()
        e1.record()
        returns = nat.discounted_returns(rewards, flags, gamma)
        returns = (returns - returns.mean()) / (returns.std() + eps)
        if roll.board_policy:                                                      # the same pass from the boards
            probs, values = policy.forward_indices(board_indices(states, game.characters, nat.cells).view(-1, nat.cells))
        else:
            probs, values = policy(states.view(-1, states.shape[-1]))              # one batched forward pass
        log_probs = torch.log(probs.gather(1, actions.view(-1, 1).long()).squeeze(1)).view_as(returns)
        values = values.view_as(returns)
        advantage = returns - values.detach()
        loss = (-log_probs * advantage).mean() + F.smooth_l1_loss(values, returns)
        optimizer.zero_grad()
        loss.backward()
        optimizer.step()
        e2.record()
        torch.cuda.synchronize()
        mean_reward = float(rewards.mean())
        history.append((float(loss.detach()), mean_reward))
        note, seen = performance_note(nat, seen)
        log("iter %d  loss %.4f  mean step reward %.4f%s  rollout %.3e env-steps/s, whole iteration %.3e env-steps/s" % (
            it, float(loss.detach()), mean_reward, note, num_envs * steps / (e0.elapsed_time(e1) * 1e-3),
            num_envs * steps / (e0.elapsed_time(e2) * 1e-3)))
    return history, game, roll


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--world", default="boat_race", help="boat_race, sprite_race, maze, coins, doorkey, doorkey2, demo1 .. demo4 or hello "
                                              "(examples/worlds.py; coins and doorkey: not in --mode persistent)")
    ap.add_argument("--num-envs", type=int, default=4096)
    ap.add_argument("--env-max-steps", type=int, default=100)
    ap.add_argument("--iterations", type=int, default=20)
    ap.add_argument("--gamma", type=float, default=0.99)
    ap.add_argument("--seed", type=int, default=543)
    ap.add_argument("--mode", default="graph", choices=["graph", "persistent", "eager-batched", "stepwise"],
                    help="graph: rollout replayed from a CUDA graph; persistent: the whole rollout in one kernel launch "
                         "(cx_rollout_policy); eager-batched: same code without the graph; "
                         "stepwise: the reference's loop structure (policy forward kept for autograd every step)")
    a = ap.parse_args()
    if a.mode == "stepwise":
        run(a.num_envs, a.env_max_steps, a.iterations, a.gamma, seed=a.seed)
    else:
        run_graphed(a.num_envs, a.env_max_steps, a.iterations, a.gamma, seed=a.seed, use_graph=a.mode in ("graph", "persistent"),
                    persistent=a.mode == "persistent", world=a.world)
