"""What a sprite agent that walls stop costs (examples/worlds.py `Runner`, PyColab's MazeWalker).

  maze          the sprite agent against its twin with a `Walker` drape as agent (the same game, the same single-agent
                kernels), at 65,536 and 2^20 envs;
  sprite_race   cx_rollout_policy at 4,096 envs against boat_race (its drape twin);
  stamp         a sprite agent painted before the first drape (it stamps the backdrop, so the game runs on the generic
                kernels) with its walls, against the same world with a sprite that walls do not stop.  Before sprites
                could have walls, only the unblocked one compiled: it is the "before" figure, and it runs the
                table-driven step that it ran then.

cx_rollout: STEPS env-batch steps as fused launches of CHUNK steps, episode limit 100 + auto reset, uniform random
actions; the games of one comparison alternate in one process, REPS repetitions each; times are CUDA events around
the whole window after warm-up.  cx_rollout_policy: POLICY_STEPS-step launches of a 32-unit policy.
Prints one JSON line per measurement; `--out FILE` writes the whole result as JSON."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from campx_b200 import things
from campx_b200.ascii_art import Partial, ascii_art_to_game
from examples.worlds import Runner, make_world
from scripts.pickup_time import card, timed_ms

STEPS, CHUNK, REPS, LIMIT, POLICY_STEPS = 1000, 20, 5, 100, 100
STAMP_ART = ['######', '#A ~ #', '# #  #', '#~   #', '######']


def make(kind, n):
    kw = dict(num_envs=n, max_episode_steps=LIMIT, track_returns=True, verify=False)
    if kind == "maze":
        game = make_world("maze", **kw)
    elif kind == "maze_drape_twin":
        game = make_world("maze", agent="drape", **kw)
    elif kind in ("sprite_race", "boat_race"):
        game = make_world(kind, **kw)
    else:
        walls = "#~" if kind == "stamp_blocked" else ""
        game = ascii_art_to_game(STAMP_ART, ' ', sprites={'A': Partial(Runner, walls=walls, per_step=0.5)},
                                 drapes={'#': things.FixedDrape}, z_order='A#', **kw)
    game.its_showtime()
    return game


def rollout_case(kind, n):
    game = make(kind, n)
    nat = game.native
    actions = [nat.fill_actions(CHUNK, seed=543, t0=i * CHUNK) for i in range(4)]
    outs = [nat.alloc_outputs(CHUNK) for _ in range(2)]

    def issue(i):
        nat.rollout(actions[i % 4], *outs[i % 2])
    for i in range(6):
        issue(i)
    return game, issue, STEPS // CHUNK, STEPS


def policy_case(kind, n):
    game = make(kind, n)
    nat = game.native
    gen = torch.Generator(device="cuda").manual_seed(3)
    feat = nat.n_chars * nat.cells
    w = (0.1 * torch.randn((feat, 32), generator=gen, device="cuda"), 0.1 * torch.randn(32, generator=gen, device="cuda"),
         0.1 * torch.randn((nat.n_actions, 32), generator=gen, device="cuda"),
         0.1 * torch.randn(nat.n_actions, generator=gen, device="cuda"))
    states = torch.empty((POLICY_STEPS + 1, n, feat), dtype=torch.float32, device="cuda")
    acts = torch.empty((POLICY_STEPS, n), dtype=torch.uint8, device="cuda")
    reward = torch.empty((POLICY_STEPS, n), dtype=torch.float32, device="cuda")
    flags = torch.empty((POLICY_STEPS, n), dtype=torch.uint8, device="cuda")

    def issue(i):
        nat.rollout_policy(POLICY_STEPS, *w, 11, states, acts, reward, flags, step_offset=i * POLICY_STEPS)
    for i in range(3):
        issue(i)
    return game, issue, 10, 10 * POLICY_STEPS


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=REPS)
    ap.add_argument("--out")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    result = {"card": card(), "steps": STEPS, "chunk": CHUNK, "episode_limit": LIMIT, "cases": []}
    plan = [(rollout_case, ("maze", "maze_drape_twin"), 65536), (rollout_case, ("maze", "maze_drape_twin"), 1 << 20),
            (policy_case, ("sprite_race", "boat_race"), 4096),
            (rollout_case, ("stamp_blocked", "stamp_unblocked"), 65536)]
    for make_case, kinds, n in plan:
        games = {k: make_case(k, n) for k in kinds}
        ms = {k: [] for k in kinds}
        for _ in range(args.reps):
            for k, (game, issue, launches, steps) in games.items():   # alternating in one process
                ms[k].append(timed_ms(issue, launches))
        for k, (game, issue, launches, steps) in games.items():
            best = min(ms[k])
            row = {"game": k, "entry": "cx_rollout_policy" if make_case is policy_case else "cx_rollout", "envs": n,
                   "path": int(game.native.info.path), "ms": [round(x, 3) for x in ms[k]], "best_ms": round(best, 3),
                   "env_steps_per_s": n * steps / (best / 1e3)}
            print(json.dumps(row), flush=True)
            result["cases"].append(row)
        del games
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
