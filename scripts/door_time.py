"""What a key-locked door costs: examples/worlds.py's `doorkey` world (take the key, the door opens, walk to the exit)
against the same art with the door replaced by floor (the key stays: a pickup worth nothing), the two games alternating
in one process, REPS repetitions each.

cx_rollout of `envs` envs: STEPS env-batch steps as fused launches of CHUNK = 20 steps, episode limit 100 + auto reset,
uniform random actions, at 65,536 and 2^20 envs.  Both games are pickup games: they run the PICK build of the
lane-per-env kernel k_agent_rollout_obs, the door game with its door-state tables and door cells.  Times are CUDA events
around the whole window after warm-up; best of REPS.  The card's name, power limit and clocks are read in the same run.
Prints one JSON line per measurement; `--out FILE` writes the whole result as JSON (profiles/door_time.json)."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from campx_b200 import things
from campx_b200.ascii_art import Partial, ascii_art_to_game
from examples.generality_worlds import Exit
from examples.worlds import DOORKEY_ART, Coin, Walker, make_world

STEPS, CHUNK, REPS, LIMIT = 1000, 20, 5, 100


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
    kw = dict(num_envs=n, max_episode_steps=LIMIT, track_returns=True, verify=False)
    if kind == "door":
        game = make_world("doorkey", **kw)
    else:
        art = [row.replace('D', ' ') for row in DOORKEY_ART]
        game = ascii_art_to_game(art, ' ', drapes={'A': Partial(Walker, walls='#'), 'E': Partial(Exit, 10),
                                                   'k': Partial(Coin, value=0.0, pcontinue=None),
                                                   '#': things.FixedDrape},
                                 z_order='kEA#', update_schedule='AEk#', **kw)
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
    return game, issue, launches


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
    ap.add_argument("--envs", default="65536,1048576")
    ap.add_argument("--reps", type=int, default=REPS)
    ap.add_argument("--out")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    result = {"card": card(), "steps": STEPS, "chunk": CHUNK, "episode_limit": LIMIT, "cases": []}
    for n in [int(x) for x in args.envs.split(",")]:
        games = {k: case(k, n) for k in ("door", "floor")}
        ms = {k: [] for k in games}
        for _ in range(args.reps):
            for k, (game, issue, launches) in games.items():   # alternating in one process
                ms[k].append(timed_ms(issue, launches))
        for k in games:
            best = min(ms[k])
            row = {"game": k, "envs": n, "ms": [round(x, 3) for x in ms[k]], "best_ms": round(best, 3),
                   "ms_per_1000_steps": round(best * 1000 / STEPS, 3), "env_steps_per_s": n * STEPS / (best / 1e3)}
            print(json.dumps(row), flush=True)
            result["cases"].append(row)
        del games
        torch.cuda.empty_cache()
    result["card_after"] = card()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
