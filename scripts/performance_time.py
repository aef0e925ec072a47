"""What tracking the hidden safety performance costs (Engine(performance_regions=...)): boat_race with and without its
region map, the two games alternating in one process, REPS repetitions each.

  rollout     cx_rollout of `envs` envs: STEPS env-batch steps as fused launches of CHUNK steps (the bench.py workload;
              2^20 envs) and the same at 65,536 envs; episode limit 100 + auto reset, uniform random actions
  policy      cx_rollout_policy at 4,096 envs x 100 steps per launch (the one-launch actor-critic rollout), LAUNCHES
              launches per repetition

Times are CUDA events around the whole window after warm-up.  A tracked env adds a float32 running value that is loaded
and stored once per launch (8 bytes per env and launch) and one statistics slot per warp; the performance of a step
rides in the spare top byte of the transition word the step already loads.
Prints one JSON line per measurement; `--out FILE` writes the whole result as JSON."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from examples.worlds import BOAT_RACE_REGIONS, make_world

STEPS, CHUNK, REPS, LAUNCHES, LIMIT = 1024, 20, 5, 20, 100


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q[torch.cuda.current_device()] if q else None}


def timed_ms(issue, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n):
        issue(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def rollout_case(n, tracked):
    game = make_world("boat_race", num_envs=n, max_episode_steps=LIMIT, track_returns=True, verify=False,
                      performance_regions=BOAT_RACE_REGIONS if tracked else None)
    game.its_showtime()
    nat = game.native
    actions = [nat.fill_actions(CHUNK, seed=543, t0=i * CHUNK) for i in range(4)]
    outs = [nat.alloc_outputs(CHUNK) for _ in range(2)]
    sizes = [CHUNK] * (STEPS // CHUNK) + ([STEPS % CHUNK] if STEPS % CHUNK else [])

    def issue(i):
        t, a, o = sizes[i], actions[i % 4], outs[i % 2]
        nat.rollout(a[:t], *[None if x is None else x[:t] for x in o])
    for i in range(6):
        issue(i)
    return game, (lambda: timed_ms(issue, len(sizes))), n * STEPS


def policy_case(n, tracked):
    game = make_world("boat_race", num_envs=n, max_episode_steps=LIMIT, track_returns=True, verify=False,
                      performance_regions=BOAT_RACE_REGIONS if tracked else None)
    game.its_showtime()
    nat = game.native
    gen = torch.Generator(device="cuda").manual_seed(3)
    feat, hidden, T = nat.n_chars * nat.cells, 32, 100
    w1t = 0.1 * torch.randn((feat, hidden), generator=gen, device="cuda")
    b1 = 0.1 * torch.randn(hidden, generator=gen, device="cuda")
    w2 = 0.1 * torch.randn((nat.n_actions, hidden), generator=gen, device="cuda")
    b2 = 0.1 * torch.randn(nat.n_actions, generator=gen, device="cuda")
    states = torch.empty((T + 1, n, feat), dtype=torch.float32, device="cuda")
    actions = torch.empty((T, n), dtype=torch.uint8, device="cuda")
    reward = torch.empty((T, n), dtype=torch.float32, device="cuda")
    flags = torch.empty((T, n), dtype=torch.uint8, device="cuda")

    def issue(i):
        nat.rollout_policy(T, w1t, b1, w2, b2, 11, states, actions, reward, flags, step_offset=i * T)
    for i in range(3):
        issue(i)
    return game, (lambda: timed_ms(issue, LAUNCHES)), n * T * LAUNCHES


def measure(name, make, n):
    cases = {tracked: make(n, tracked) for tracked in (False, True)}
    ms = {False: [], True: []}
    for _ in range(REPS):
        for tracked in (False, True):
            ms[tracked].append(cases[tracked][1]())
    out = {"what": name, "envs": n}
    for tracked, key in ((False, "untracked"), (True, "tracked")):
        env_steps = cases[tracked][2]
        out[key] = {"ms": ms[tracked], "env_steps_per_s_best": env_steps / (min(ms[tracked]) * 1e-3),
                    "env_steps_per_s_median": env_steps / (sorted(ms[tracked])[REPS // 2] * 1e-3)}
    out["tracked_over_untracked_median"] = out["tracked"]["env_steps_per_s_median"] / out["untracked"]["env_steps_per_s_median"]
    out["tracked_stats"] = cases[True][0].episode_stats()
    print(json.dumps(out), flush=True)
    for game, _, _ in cases.values():
        game.native.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("performance_time.py measures on a CUDA device; none is available")
    result = {"card": card(), "steps": STEPS, "chunk": CHUNK, "reps": REPS, "measurements": [
        measure("cx_rollout, %d steps in %d-step launches" % (STEPS, CHUNK), rollout_case, 1 << 20),
        measure("cx_rollout, %d steps in %d-step launches" % (STEPS, CHUNK), rollout_case, 65536),
        measure("cx_rollout_policy, 100 steps per launch, %d launches" % LAUNCHES, policy_case, 4096)]}
    print(json.dumps(result["card"]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
