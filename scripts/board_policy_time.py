"""Development aid: cx_policy_sample_board (the policy read off the uint8 board) against the routes it replaces, and the
Hello World actor-critic rollout of examples/actor_critic_batched.py.

Every kernel time is CUDA events around a CUDA graph of LAUNCHES captured calls, after warm-up, divided by LAUNCHES.
  board     cx_policy_sample_board on boards [n, rows, cols] uint8
  planes    cx_policy_sample on float32 planes made beforehand (boat_race: the input cx_step_observations writes)
  l2p       cx_layers_from_board_f32 + cx_policy_sample (boat_race: planes made from the same boards)
  torch     cx_layers_from_board_f32 + Policy.action_logits (cuBLAS) + cx_sample_actions (Hello World: the route a user
            had before cx_policy_sample_board)
Bytes are counted from shapes.  board: the boards, plus the W1^T rows the set-input walk gathers -- one 128-byte row
(16 bytes per warp) per set input, at most `cells` per env -- from shared memory when W1^T is staged there (boat_race),
otherwise from global memory, where L1 / L2 serve them (Hello World: 419 KB of W1^T); how much of it L2 serves is not
measured.
Prints one JSON line per measurement; `--out FILE` also writes them as a JSON list."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from examples.actor_critic_batched import Policy, run_graphed
from examples.worlds import make_world

LAUNCHES = 50


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q[torch.cuda.current_device()] if q else None}


def graph_us(fn, reps):
    """us per call: `fn` captured LAUNCHES times in one graph, replayed `reps` times after warm-up."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(LAUNCHES):
            fn()
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * LAUNCHES)


def kernels(world, n, reps):
    game = make_world(world, num_envs=n, max_episode_steps=100)
    game.its_showtime()
    nat = game.native
    board = game.rollout(nat.fill_actions(7, seed=3))[0][-1].contiguous()
    feat = nat.n_chars * nat.cells
    torch.manual_seed(1)
    pol = Policy(feat, n_actions=nat.n_actions).cuda()
    w1t = pol.affine1.weight.detach().t().contiguous()
    b1, w2, b2 = pol.affine1.bias.detach(), pol.action_head.weight.detach(), pol.action_head.bias.detach()
    acts = torch.empty(n, dtype=torch.uint8, device="cuda")
    planes = torch.empty((n, nat.n_chars, nat.rows, nat.cols), dtype=torch.float32, device="cuda")
    flat = planes.view(n, -1)
    ctas = (n + 31) // 32
    res = {"world": world, "envs": n, "inputs": feat, "launches_per_graph": LAUNCHES,
           "w1t_bytes": feat * 32 * 4, "board_bytes": n * nat.cells, "plane_bytes": n * feat * 4}
    routes = {"board": lambda: nat.policy_sample_board(board, w1t, b1, w2, b2, 7, out=acts)}
    if world == "boat_race":
        nat.layers_from_board(board, out=planes, dtype=torch.float32)
        routes["planes"] = lambda: nat.policy_sample(flat, w1t, b1, w2, b2, 7, out=acts)
        routes["l2p"] = lambda: (nat.layers_from_board(board, out=planes, dtype=torch.float32),
                                 nat.policy_sample(flat, w1t, b1, w2, b2, 7, out=acts))

    def torch_route():
        nat.layers_from_board(board, out=planes, dtype=torch.float32)
        nat.sample_actions(pol.action_logits(flat), 7, logits=True, out=acts)
    routes["torch"] = torch_route
    with torch.no_grad():
        for name, fn in routes.items():
            res[name + "_us"] = round(graph_us(fn, reps), 3)
    # W1^T rows the set-input walk gathers: 128 B (8 warps x 16 B) per set input; staging, where W1^T fits shared
    # memory, adds feat * 128 B per CTA
    set_inputs = int(nat.layers_from_board(board).sum())
    res["board_set_inputs"] = set_inputs
    res["board_w1t_bytes_per_launch"] = set_inputs * 128
    res["board_w1t_staged_bytes_per_launch"] = ctas * feat * 128
    res["board_w1t_from"] = "shared memory (staged from L2 once per CTA)" if (
        8 * 8 * 33 * 4 + feat * 128 + 32 * 4 * (((nat.cells + 3) // 4) | 1) + 256 + 8 * nat.n_chars * 128 + 128
        + nat.cells * 128) <= 100 * 1024 else "L1 / L2 (global loads)"
    us = res["board_us"]
    res["board_GBps_boards_only"] = round(res["board_bytes"] / us * 1e-3, 1)
    res["board_GBps_incl_w1t"] = round((res["board_bytes"] + res["board_w1t_bytes_per_launch"]) / us * 1e-3, 1)
    res["board_envs_per_s"] = round(n / us * 1e6, 1)
    return res


def rollout(n, steps, iterations):
    lines = []
    history, game, roll = run_graphed(world="hello", num_envs=n, steps=steps, iterations=iterations, log=lines.append)
    return {"world": "hello", "what": "actor_critic_batched --world hello --mode graph", "envs": n, "steps": steps,
            "step_kernel": roll.step_kernel, "log": lines}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="4096,65536,262144")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = [dict(card(), what="card")]
    print(json.dumps(out[0]), flush=True)
    for world in ("boat_race", "hello"):
        for n in (int(s) for s in a.sizes.split(",")):
            out.append(kernels(world, n, a.reps))
            print(json.dumps(out[-1]), flush=True)
    out.append(rollout(4096, 100, 6))
    print(json.dumps(out[-1]), flush=True)
    out.append(dict(card(), what="card (after)"))
    print(json.dumps(out[-1]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
