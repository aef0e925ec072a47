"""What collectible items cost: examples/worlds.py's `coins` world (ten `$` pickups, the episode ends with the last one)
against the same art with the coins as static reward tiles (`Walker(treasures='$')`: pays on every entry, never
disappears), the two games alternating in one process, REPS repetitions each.

cx_rollout of `envs` envs: STEPS env-batch steps as fused launches of CHUNK steps, episode limit 100 + auto reset,
uniform random actions, at 65,536, 2^18 and 2^20 envs.  Pickup games always run the PICK build of the lane-per-env
kernel k_agent_rollout_obs; the static-tile game takes its automatic route.  Times are CUDA events around the whole
window after warm-up; the share of peak is the algorithmic bytes (action, reward, discount, flags and board of every
env-step) over the time, against the measured copy peak of 6,534.1 GB/s (DESIGN section 5).
Prints one JSON line per measurement; `--out FILE` writes the whole result as JSON."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from campx_b200 import things
from campx_b200.ascii_art import Partial, ascii_art_to_game
from examples.worlds import COINS_ART, Walker, make_world

STEPS, CHUNK, REPS, LIMIT = 1000, 20, 5, 100
PEAK_GBS = 6534.1


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    lines = q.splitlines()
    return {"device": torch.cuda.get_device_name(),
            "nvidia_smi name, power.limit, clocks.sm, clocks.max.sm": lines[torch.cuda.current_device()] if lines else None}


def make(kind, n):
    if kind == "pickups":
        game = make_world("coins", num_envs=n, max_episode_steps=LIMIT, track_returns=True, verify=False)
    else:
        game = ascii_art_to_game(COINS_ART, ' ', drapes={'A': Partial(Walker, walls='#', treasures='$'),
                                                         '$': things.FixedDrape, '#': things.FixedDrape},
                                 z_order='$A#', update_schedule='A$#', num_envs=n, max_episode_steps=LIMIT,
                                 track_returns=True, verify=False)
    game.its_showtime()
    return game


def case(kind, n):
    game = make(kind, n)
    nat = game.native
    actions = [nat.fill_actions(CHUNK, seed=543, t0=i * CHUNK) for i in range(4)]
    outs = [nat.alloc_outputs(CHUNK) for _ in range(2)]
    launches = STEPS // CHUNK

    def issue(i):
        nat.rollout(actions[i % 4], *outs[i % 2])
    for i in range(6):
        issue(i)
    per_step = 1 + 4 + 1 + nat.cells + (4 if outs[0][3] is not None else 0)
    return game, issue, launches, per_step


def timed_ms(issue, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n):
        issue(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="65536,262144,1048576")
    ap.add_argument("--reps", type=int, default=REPS)
    ap.add_argument("--out")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    result = {"card": card(), "steps": STEPS, "chunk": CHUNK, "episode_limit": LIMIT, "copy_peak_GBs": PEAK_GBS,
              "cases": []}
    for n in [int(x) for x in args.envs.split(",")]:
        games = {k: case(k, n) for k in ("pickups", "static_tiles")}
        ms = {k: [] for k in games}
        for _ in range(args.reps):
            for k, (game, issue, launches, _) in games.items():   # alternating in one process
                ms[k].append(timed_ms(issue, launches))
        for k, (game, issue, launches, per_step) in games.items():
            best = min(ms[k])
            rate = n * STEPS / (best / 1e3)
            row = {"game": k, "envs": n, "ms": [round(x, 3) for x in ms[k]], "best_ms": round(best, 3),
                   "env_steps_per_s": rate, "bytes_per_env_step": per_step,
                   "share_of_copy_peak": rate * per_step / (PEAK_GBS * 1e9)}
            print(json.dumps(row), flush=True)
            result["cases"].append(row)
        del games
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
