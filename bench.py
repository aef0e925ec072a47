#!/usr/bin/env python
"""Benchmark of the batched Engine.play() hot path: boat_race, 2^20 environments per GPU.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W

A "step" is one Engine.play() over the whole environment batch (N_envs env-steps per GPU).  Steps are issued
as fused `cx_rollout` launches of `--chunk` steps each (state stays on chip inside a launch); inputs (uint8
action indices, generated beforehand with the library's Philox kernel) are resident in HBM when the timed
region starts, and every env-step writes its full observation contract (board 25 B, reward f32, flags u8)
to HBM.  One launch writes ~630 MB, far more than the 126 MB L2, and consecutive launches alternate between
two output buffers.

How the timed region is built (so that it measures the kernels, not the host's launch path):
  * it holds exactly --steps env-batch steps (fused launches of --chunk steps, plus one shorter launch for a
    remainder); value = envs * K / time.  A step of 2^20 envs takes ~5 us, so a K of a few hundred or more
    keeps the edges of the window small against the work inside it;
  * the region starts on a BUSY stream: a few untimed launches are queued first and the start event is
    recorded behind them, so host launch latency never sits inside the event window;
  * the NVML clock sampler polls every 50 ms.

`--dump-outputs DIR` writes what the timed launches returned for their last step (see `dump_outputs`); the
inputs depend only on the arguments, so two builds run with the same arguments can be compared array for array.

Before anything is timed every rank replays a sample of its own environments through the CPU oracle
(`parity_check`), and the JSON line carries a `configs` block with the other BASELINE.json configurations
(Hello World / Demo 1 at 65,536 envs, Demo 2 / Demo 4 at 2^20, the 4,096-env actor-critic rollout), each
with its own event timing, algorithmic bytes, roofline fraction and sampled oracle check.

JSON line keys follow the driver contract; see DESIGN.md "Measurement" for how each number is taken.
"""
import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORLD = "boat_race"
EPISODE_LIMIT = 100          # examples/actor_critic.py:56
SEED = 543                   # examples/actor_critic.py:26
PARITY_ENVS = 64             # SURVEY 8(d): first 64 envs of each rank ...
PARITY_STEPS = 1000          # ... first 1,000 steps (ten episodes: the auto-reset at step 100 is crossed nine times)
CONFIG_PARITY_STEPS = 128    # the `configs` entries: a shorter replay per config


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1024, help="env-batch steps inside the timed region")
    ap.add_argument("--warmup", type=int, default=64)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=1 << 20, help="environments per GPU")
    ap.add_argument("--chunk", type=int, default=20,
                    help="env-batch steps fused per kernel launch (20: measured optimum of k_agent_rollout at 2^20 envs, "
                         "DESIGN.md section 5.1; longer rollouts are split into such launches by the library anyway)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned (board, reward, flags and any discount) to DIR "
                         "as float32 .npy files")
    ap.add_argument("--e2e-steps", type=int, default=64)
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="budget of each cpu_baseline leg")
    ap.add_argument("--obs-reps", type=int, default=8,
                    help="launches of the secondary board+layered-board measurement (0: skip it)")
    ap.add_argument("--parity-steps", type=int, default=PARITY_STEPS,
                    help="steps every rank replays through the CPU oracle before timing (profiler passes shorten it)")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` block (other BASELINE configs)")
    ap.add_argument("--reference-root", default=os.environ.get("CAMPX_REFERENCE_ROOT", ""),
                    help="directory holding the unmodified reference (campx/ + examples/): the CPU legs then ALSO "
                         "time the reference's own Engine.play under oracle/shim.py.  Never read unless given; "
                         "baseline/_ref is picked up when it exists.")
    return ap.parse_args()


# --------------------------------------------------------------------------------------------------
# CPU arm: Engine.play of the reference on the host cores, one env per object.
#   kind "port"      oracle/campx_oracle.py, the numpy restatement (always available)
#   kind "reference" the UNMODIFIED reference package under oracle/shim.py (only where its tree exists)
# --------------------------------------------------------------------------------------------------

def reference_root(args):
    for cand in (args.reference_root, os.path.join(ROOT, "baseline", "_ref")):
        if cand and os.path.isdir(os.path.join(cand, "campx")) and \
                os.path.isfile(os.path.join(cand, "examples", "boat_race.py")):
            return cand
    return None


def _port_factory():
    from oracle import campx_oracle as O

    def make():
        w = O.World(WORLD)
        return lambda a: w.step(a)
    return make


def _reference_factory(root):
    import torch
    from oracle import shim
    shim.install(root)
    torch.set_num_threads(1)                              # SURVEY 8(d): one core per process
    import boat_race as ref_boat_race                      # the reference's examples/boat_race.py, unmodified
    onehots = [torch.eye(5)[i] for i in range(5)]          # FloatTensor one-hot actions (boat_race.py:26)

    def make():
        game, _, _, _ = ref_boat_race.make_game()
        return lambda a: game.play(onehots[a])
    return make


def _cpu_worker(job):
    n_envs, warm, steps, seed, kind, root = job
    import numpy as np
    make = _reference_factory(root) if kind == "reference" else _port_factory()
    rng = np.random.Generator(np.random.PCG64(seed))
    envs = [make() for _ in range(n_envs)]
    age = [0] * n_envs

    def batch_step():
        acts = rng.integers(0, 5, size=n_envs)
        for i in range(n_envs):
            envs[i](int(acts[i]))
            age[i] += 1
            if age[i] >= EPISODE_LIMIT:          # a fresh make_game() per episode (actor_critic.py:146)
                envs[i] = make()
                age[i] = 0

    for _ in range(warm):
        batch_step()
    t0 = time.perf_counter()
    for _ in range(steps):
        batch_step()
    return n_envs * steps, time.perf_counter() - t0


def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_rate(steps, warm, budget_s, kind="port", root=None, cores=None):
    """env-steps/s of the CPU Engine.play: (i) one process on one core, (ii) `cores` independent processes.

    Each of `steps` steps advances a bounded sample of environments, sized from a calibration run so that
    each leg fits `budget_s` seconds.  Returns a `cpu_baseline` dict (value = the all-cores figure)."""
    import multiprocessing as mp
    if cores is None:
        cores = host_cores()
    ctx = mp.get_context("fork")
    what = ("oracle/campx_oracle.py (numpy port of the reference's Engine.play)" if kind == "port" else
            "the unmodified reference Engine.play under oracle/shim.py, torch.set_num_threads(1)")

    def run(procs, per_proc, w, s):
        jobs = [(per_proc, w, s, SEED + i, kind, root) for i in range(procs)]
        with ctx.Pool(procs) as pool:                      # a forked child per leg: the parent never imports the oracle
            res = pool.map(_cpu_worker, jobs)
        return sum(r[0] for r in res) / max(r[1] for r in res), max(r[1] for r in res)

    cal, _ = run(1, 2, 1, 20)                              # calibration, one core
    per_one = int(max(1, min(256, cal * min(budget_s, 4.0) / max(1, steps + warm))))
    one, _ = run(1, per_one, warm, steps)
    per_core = int(max(1, min(256, one * budget_s / max(1, steps + warm))))
    allc, elapsed = run(cores, per_core, warm, steps)
    sample = "%d procs x %d envs x %d steps of %s, episode rebuilt every %d steps; %s" % (
        cores, per_core, steps, WORLD, EPISODE_LIMIT, what)
    return {"value": allc, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample,
            "one_core": {"value": one, "unit": "env-steps/s", "cores": 1,
                         "sample": "1 proc x %d envs x %d steps" % (per_one, steps)}}, elapsed


def cpu_baseline(args, steps, warm, budget_s):
    """`cpu_baseline` of the JSON line: the port always; the shimmed reference next to it where its tree is given."""
    cpu, elapsed = cpu_rate(steps, warm, budget_s, "port")
    root = reference_root(args)
    if root is not None:
        try:
            ref, elapsed_ref = cpu_rate(steps, warm, budget_s, "reference", root)
            ref["port"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "one_core")}
            return ref, elapsed_ref
        except Exception as exc:                           # an unusable tree must not cost the bench line
            cpu["reference_error"] = repr(exc)
    return cpu, elapsed


def workload_config(envs, world, chunk):
    """`config` of the JSON line; identical for both arms (the reference arm times a bounded sample of it)."""
    per_step = 1 + 4 + 1 + 25
    return {"workload": "boat_race 5x5 (examples/worlds.py == reference examples/boat_race.py), "
                        "2^20 envs per GPU, uniform random actions, episode limit 100 + auto reset",
            "envs_per_gpu": envs, "total_envs": world * envs, "fused_steps_per_launch": chunk,
            "observation_contract": "board u8[25] + reward f32 + flags u8 per env-step",
            "l2_policy": "outputs larger than L2: each launch writes %.0f MB, two alternating output "
                         "buffers" % (envs * chunk * (per_step - 1) / 1e6),
            "parallelism": "env-sharded x%d, no step-path collective" % world}


def run_reference(args, rank):
    if rank != 0:
        return
    steps = max(1, min(args.steps, 2000))
    warm = max(0, min(args.warmup, 20))
    cpu, elapsed = cpu_baseline(args, steps, warm, budget_s=30.0)
    value = cpu["value"]
    line = {
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": elapsed * 1e3 / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.envs, max(1, args.gpus), max(1, args.chunk)),
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------

class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the benchmark runs (every 50 ms:
    rare enough not to disturb the launch thread, frequent enough for a handful of samples per timed region)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index, period=0.05):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.active = False          # only samples taken while `active` count as "under load"
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def sample_once(self):
        nv = self.nv
        mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        self.samples.append(mhz)
        for bit, name in self.REASONS.items():
            if mask & bit:
                self.reasons.add(name)

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            if self.active:
                try:
                    self.sample_once()
                except Exception:
                    pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=1.0)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s), "period_ms": self.period * 1e3}


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------

def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def ncu_traffic(key):
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return json.load(f).get(key)
    except Exception:
        return None


def oracle_check(world, nat, make_actions, launch, envs, steps, T, limit=EPISODE_LIMIT, layers=True):
    """Replay `envs` (indices into this game's batch) through the CPU oracle for `steps` steps and require
    board, every layer, reward, discount and the done flags to be EQUAL to what the kernels wrote.

    The game must be in its its_showtime state.  `make_actions(i)` -> uint8 [T, n] device actions of launch i,
    `launch(a, out)` runs them.  Returns (ok, first mismatch or None)."""
    import numpy as np
    import torch
    from campx_b200 import _native as N
    from oracle import campx_oracle as O                  # the checker: never timed, never on the product path

    idx = torch.as_tensor(list(envs), dtype=torch.long, device=nat.device)
    got = {"a": [], "b": [], "r": [], "f": [], "d": [], "l": []}
    out = nat.alloc_outputs(T, discount=nat.wants_discount)
    for i in range((steps + T - 1) // T):
        a = make_actions(i)
        launch(a, out)
        board, reward, flags, disc = out
        sel = board[:, idx].contiguous()
        got["a"].append(a[:, idx].cpu().numpy())
        got["b"].append(sel.cpu().numpy())
        got["r"].append(reward[:, idx].cpu().numpy())
        got["f"].append(flags[:, idx].cpu().numpy())
        if disc is not None:
            got["d"].append(disc[:, idx].cpu().numpy())
        if layers:
            got["l"].append(nat.layers_from_board(sel).cpu().numpy())
    cat = {k: (np.concatenate(v) if v else None) for k, v in got.items()}
    chars = list(nat.spec.chars)                           # canonical channel order (sorted by code point)
    for j, env in enumerate(envs):
        for t, (o, rew, dsc, term, trunc, eng) in enumerate(
                O.rollout(world, cat["a"][:steps, j], rebuild_on_done=True, max_episode_steps=limit)):
            f = int(cat["f"][t, j])
            ok = np.array_equal(cat["b"][t, j], np.asarray(o.board).astype(np.uint8))
            ok = ok and (0.0 if rew is None else float(rew)) == float(cat["r"][t, j])
            ok = ok and (rew is None) == bool(f & N.CX_FLAG_REWARD_NONE)
            ok = ok and term == bool(f & N.CX_FLAG_TERMINATED) and trunc == bool(f & N.CX_FLAG_TRUNCATED)
            if cat["d"] is not None:
                ok = ok and float(dsc) == float(cat["d"][t, j])
            if layers and ok:
                for k, ch in enumerate(chars):
                    ok = ok and np.array_equal(cat["l"][t, j, k], np.asarray(o.layers[ch]).astype(np.uint8))
            if not ok:
                return False, {"env": int(env), "step": t}
    return True, None


def device_time_ms(issue, lead, count):
    """Event time of `count` launches issued back to back behind `lead` untimed ones (busy stream at the start)."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    for i in range(lead):
        issue(i)
    e0.record()
    for i in range(count):
        issue(lead + i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


DUMP_BYTES = 60 * 10 ** 6          # --dump-outputs writes at most this much array data (plus .npy headers)


def dump_outputs(path, out, t):
    """--dump-outputs: step `t` of the rollout buffers `out` (board, reward, flags, discount or None), i.e. what a
    caller of Engine.rollout receives for that step, as float32 DIR/<name>.npy.  When every env would exceed
    DUMP_BYTES, a fixed sample of envs (PCG64 seeded with SEED, sorted) is written; env_index.npy (float64)
    names the envs, row for row."""
    import numpy as np
    import torch
    board, reward, flags, disc = out
    arrays = {"board": board[t], "reward": reward[t], "flags": flags[t]}
    if disc is not None:
        arrays["discount"] = disc[t]
    n = board.shape[1]
    per_env = 8 + sum(4 * a[0].numel() for a in arrays.values())
    if n * per_env <= DUMP_BYTES:
        idx = np.arange(n)
    else:
        idx = np.sort(np.random.Generator(np.random.PCG64(SEED)).choice(n, DUMP_BYTES // per_env, replace=False))
    sel = torch.as_tensor(idx, device=board.device)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "env_index.npy"), idx.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a[sel].float().cpu().numpy())


def hello_actions(nat, T, seed):
    """SURVEY 8(d): Hello World actions uniform over 0..3 plus 1% quit (action 4)."""
    import torch
    a = nat.fill_actions(T, seed=seed)                         # uniform over 0..4
    keep_quit = torch.rand(a.shape, device=a.device) < 0.05    # 0.2 * 0.05 = 1% quit
    repl = torch.randint(0, 4, a.shape, device=a.device, dtype=torch.uint8)
    return torch.where((a == 4) & ~keep_quit, repl, a).contiguous()


def measure_config(world_name, n, T, peak, min_ms, sampler, kernel):
    """One BASELINE config through the public API: sampled oracle check, then CUDA-graph replays of a ring of
    fused T-step launches (outputs of the ring > L2) timed with CUDA events over >= min_ms."""
    import torch
    from examples.worlds import make_world

    game = make_world(world_name, num_envs=n, max_episode_steps=EPISODE_LIMIT, auto_reset=True, track_returns=True)
    game.its_showtime()
    nat = game.native
    hello = world_name == "hello"
    per_step = 1 + 4 + 1 + nat.cells + (4 if nat.wants_discount else 0)
    state_rw = 2 * nat.info.state_bytes_per_env
    make = (lambda i: hello_actions(nat, T, SEED + i)) if hello else (lambda i: nat.fill_actions(T, seed=SEED, t0=i * T))
    envs = list(range(8)) + [n // 2, n - 1]
    ok, where = oracle_check(world_name, nat, make, lambda a, o: nat.rollout(a, *o), envs, CONFIG_PARITY_STEPS, T)
    game.reset()

    ring = max(2, int(math.ceil(400e6 / (n * T * per_step))))
    bufs = [nat.alloc_outputs(T) for _ in range(ring)]
    acts = [make(100 + i) for i in range(ring)]

    per_graph = max(ring, 8)                                   # launches per graph replay (replay gaps amortised)

    def one_ring():
        for i in range(per_graph):
            nat.rollout(acts[i % ring], *bufs[i % ring])

    # small launches (tens of microseconds) are replayed from a CUDA graph so that host launch cost cannot show;
    # large ones are issued directly, back to back, so that programmatic dependent launch overlaps their seams
    # exactly as in the headline measurement
    use_graph = n * T * per_step < 3e8
    if use_graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                          # warm-up off the capture (lazy kernel configuration)
            for _ in range(2):
                one_ring()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            one_ring()
        issue = lambda i: graph.replay()
    else:
        one_ring()
        issue = lambda i: one_ring()
    pilot = device_time_ms(issue, 1, 2) / 2
    # the oracle check above kept the GPU idle for seconds: bring it back under load (clocks, caches) before timing
    device_time_ms(issue, 0, max(2, int(math.ceil(150.0 / max(pilot, 1e-3)))))
    reps = max(2, int(math.ceil(min_ms / max(pilot, 1e-3))))
    sampler.active = True
    ms = device_time_ms(issue, 1, reps)
    sampler.active = False
    launches = reps * per_graph
    env_steps = float(launches) * n * T
    alg = env_steps * per_step + float(launches) * n * state_rw
    gbs = alg / (ms * 1e-3) / 1e9
    return {"world": world_name, "envs": n, "fused_steps_per_launch": T, "launches": launches, "timed_ms": ms,
            "env_steps_per_sec": env_steps / (ms * 1e-3), "avg_launch_ms": ms / launches,
            "alg_bytes_per_env_step": per_step + state_rw / T, "achieved_gbs": gbs, "frac": gbs / peak,
            "kernel": kernel, "l2_policy": "ring of %d output buffers, %.0f MB" % (ring, ring * n * T * per_step / 1e6),
            "issue": ("CUDA graph of %d launches over the ring, replayed" if use_graph else
                      "%d direct launches over the ring per repetition, back to back (PDL)") % per_graph,
            "parity": {"envs": len(envs), "steps": CONFIG_PARITY_STEPS, "ok": bool(ok), "mismatch": where,
                       "what": "board, every layer, reward, discount, done flags == CPU oracle"}}


def measure_actor_critic(peak, min_ms, sampler):
    """BASELINE config 5: the 4,096-env actor-critic rollout on boat_race, policy on the device, whole 100-step
    rollout replayed from a CUDA graph (examples/actor_critic_batched.py; reference examples/actor_critic.py:146-173)."""
    import numpy as np
    import torch
    from campx_b200 import _native as N
    from examples.actor_critic_batched import GraphedRollout, Policy
    from examples.worlds import make_world
    from oracle import campx_oracle as O

    n, T = 4096, EPISODE_LIMIT
    torch.manual_seed(SEED)
    game = make_world(WORLD, num_envs=n, max_episode_steps=T, track_returns=True)
    game.its_showtime()
    nat = game.native
    policy = Policy(nat.n_chars * nat.cells).to(nat.device)
    roll = GraphedRollout(game, policy, T, persistent=True).capture()   # cx_rollout_policy: the whole rollout in one launch
    states, actions, rewards, flags = roll.run()
    torch.cuda.synchronize()
    # sampled oracle check: states[t] is the layered board the policy saw BEFORE action t
    a, s = actions.cpu().numpy(), states.cpu().numpy().reshape(T, n, nat.n_chars, nat.rows, nat.cols)
    r, f = rewards.cpu().numpy(), flags.cpu().numpy()
    ok, where, envs = True, None, [0, 1, 2, 3, n // 2, n - 1]
    for i in envs:
        prev = O.World(WORLD).first[0]
        for t, (o, rew, dsc, term, trunc, eng) in enumerate(O.rollout(WORLD, a[:, i], max_episode_steps=T)):
            good = np.array_equal(s[t, i], np.asarray(prev.layered_board).astype(np.float32)) and \
                float(rew) == float(r[t, i]) and trunc == bool(f[t, i] & N.CX_FLAG_TRUNCATED)
            if not good and ok:
                ok, where = False, {"env": i, "step": t}
            prev = o
    pilot = device_time_ms(lambda i: roll.run(), 1, 2) / 2
    device_time_ms(lambda i: roll.run(), 0, max(2, int(math.ceil(150.0 / max(pilot, 1e-3)))))   # back under load
    reps = max(2, int(math.ceil(min_ms / max(pilot, 1e-3))))
    sampler.active = True
    ms = device_time_ms(lambda i: roll.run(), 1, reps)
    sampler.active = False
    per_step = 1 + 4 + 1 + nat.cells + 4 * nat.n_chars * nat.cells
    env_steps = float(reps) * n * T
    gbs = env_steps * per_step / (ms * 1e-3) / 1e9
    return {"world": "boat_race actor-critic rollout (policy Linear(175,32)-ReLU-Linear(32,5) sampled on device)",
            "envs": n, "steps_per_rollout": T, "rollouts": reps, "timed_ms": ms,
            "env_steps_per_sec": env_steps / (ms * 1e-3), "us_per_env_batch_step": ms * 1e3 / (reps * T),
            "alg_bytes_per_env_step": per_step, "achieved_gbs": gbs, "frac": gbs / peak,
            "kernel": roll.step_kernel, "kernels_per_step": roll.kernels_per_step,
            "issue": "one CUDA graph per 100-step rollout (weight transpose, cx_rollout_policy, reset), replayed",
            "bound": "latency of the per-step chain policy -> sample -> play (a 4,096-env step moves 3 MB: 128 CTAs of "
                     "32 envs keep their policy input in shared memory; five / two launches per step: 1.8e8 / 3.9e8)",
            "parity": {"envs": len(envs), "steps": T, "ok": bool(ok), "mismatch": where,
                       "what": "policy input planes (f32), reward, truncation == CPU oracle on the sampled actions"}}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from campx_b200 import dist as cxdist
    from examples.worlds import make_world

    # the CPU legs fork worker processes: they run before this process touches CUDA (a forked child must not
    # inherit a CUDA context), on rank 0 of a single-GPU run only
    cpu = None
    if int(os.environ.get("RANK", "0")) == 0 and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        cpu, _ = cpu_baseline(args, steps=200, warm=5, budget_s=args.cpu_seconds)

    rank, world, local_rank = cxdist.init_from_env()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    n, T, K, W = args.envs, max(1, args.chunk), max(1, args.steps), max(args.warmup, 3)

    sampler = ClockSampler(local_rank)
    sampler.start()

    game = make_world(WORLD, num_envs=n, max_episode_steps=EPISODE_LIMIT, auto_reset=True, track_returns=True)
    game.its_showtime()                      # compiles the user-level world and uploads it
    nat = game.native
    env_offset = rank * n                    # rank r owns envs [r*n, (r+1)*n): independent Philox streams

    def barrier():
        if world > 1:
            dist.barrier()

    def reduce_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- parity first: this rank's first 64 envs (and its last one) against the CPU oracle, on THIS game and
    # THIS rank's action streams, through the same cx_rollout launches that are timed below ----
    p_envs = list(range(min(PARITY_ENVS, n))) + ([n - 1] if n > PARITY_ENVS else [])
    p_ok, p_where = oracle_check(
        WORLD, nat, lambda i: nat.fill_actions(T, seed=SEED, env_offset=env_offset, t0=i * T),
        lambda a, o: nat.rollout(a, *o), p_envs, args.parity_steps, T)
    p_all = reduce_max(0.0 if p_ok else 1.0) == 0.0
    parity = {"ranks": world, "envs": len(p_envs), "steps": args.parity_steps, "ok": bool(p_all),
              "mismatch": p_where, "kernel": "cx_rollout on this rank's %d-env batch" % n,
              "what": "per rank: first %d envs + last env, %d steps (auto-reset at %d crossed), actions from the rank's "
                      "own Philox stream (cx_fill_actions, env_offset = rank * envs); board, every layer, reward, "
                      "done flags == oracle/campx_oracle.py; MIN over ranks" % (PARITY_ENVS, args.parity_steps, EPISODE_LIMIT)}
    game.reset()                             # back to the its_showtime state, statistics zeroed

    n_act = 4
    actions = [nat.fill_actions(T, seed=SEED, env_offset=env_offset, t0=i * T) for i in range(n_act)]
    outs = [game.alloc_rollout(T) for _ in range(2)]

    def plan(total_steps):
        """total_steps env-batch steps as fused launches of T steps (+ one shorter launch for the remainder)."""
        full, rem = divmod(total_steps, T)
        return [T] * full + ([rem] if rem else [])

    def issue_factory(sizes):
        def issue(i):
            t = sizes[i]
            a, o = actions[i % n_act], outs[i % 2]
            if t == T:
                nat.rollout(a, *o)
            else:
                nat.rollout(a[:t], *[None if x is None else x[:t] for x in o])
        return issue

    lead = 6                                 # ~1 ms of queued work in front of the start event
    warm = plan(W)
    for i in range(len(warm)):               # warm-up (>= 3 steps)
        issue_factory(warm)(i)
    sizes = [T] * lead + plan(K)
    launches = len(sizes) - lead
    issue = issue_factory(sizes)

    torch.cuda.synchronize()
    barrier()
    sampler.active = True
    ms = device_time_ms(issue, lead, launches)
    sampler.active = False
    barrier()
    ms = reduce_max(ms)
    total_steps = K
    value = world * n * total_steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        last = len(sizes) - 1
        dump_outputs(args.dump_outputs, outs[last % 2], sizes[last] - 1)

    # ---- roofline of the dominant kernel (k_agent_rollout): algorithmic bytes / avg launch duration ----
    cells = nat.cells
    per_step = 1 + 4 + 1 + cells                     # action u8 + reward f32 + flags u8 + board u8[25]
    state_rw = 2 * (1 + 2 + 4)                       # per launch and env: cell u8, step u16, return f32 (r+w)
    alg_bytes_total = n * (total_steps * per_step + launches * state_rw)
    achieved = alg_bytes_total / (ms * 1e-3) / 1e9   # this rank's kernel stream; ms is the max over ranks
    peak, peak_src = measured_peak()
    t_main = sizes[lead]
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic("k_agent_rollout_track_T%d_n%d" % (t_main, n)),
                "traffic_source": "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum of one T=%d launch "
                                  "(profiles/roofline_traffic.json; a profiler pass, not this run)" % t_main,
                "kernel": "k_agent_rollout<TRACK=true,NG=1,GW=2> (64 envs per warp)", "fused_steps_per_launch": t_main,
                "alg_bytes_per_env_step": alg_bytes_total / (n * total_steps),
                "alg_bytes_per_launch": n * (t_main * per_step + state_rw), "avg_launch_ms": ms / launches,
                "launches_timed": launches, "peak_source": peak_src}
    config = workload_config(n, world, t_main)
    config.update({"timed_steps": total_steps, "timed_region_ms": ms,
                   "timing": "K steps as back-to-back fused launches (value = envs*K/time), CUDA events on the launch "
                             "stream behind %d queued untimed launches, max over ranks" % lead})

    # ---- end to end through Engine.play() with HOST buffers (H2D actions, D2H board+reward+flags) ----
    # Every step: pinned-host actions -> device, one Engine.play(), the whole result (board, reward, flags) ->
    # pinned host.  play() alternates between two output buffer sets, so the D2H of step t runs on a side
    # stream while the H2D + kernel of step t+1 run on the main stream (PCIe is full duplex); events keep a
    # buffer set from being overwritten before its copy-out has finished.
    E = max(1, args.e2e_steps)
    numa = bind_to_gpu_numa_node(local_rank)            # pinned buffers are first-touched on the GPU's own node
    h_act = torch.randint(0, 5, (E, n), dtype=torch.uint8).pin_memory()
    h_out = [(torch.empty((n, 5, 5), dtype=torch.uint8).pin_memory(), torch.empty((n,), dtype=torch.float32).pin_memory(),
              torch.empty((n,), dtype=torch.uint8).pin_memory()) for _ in range(2)]
    d_act = [torch.empty((n,), dtype=torch.uint8, device=dev) for _ in range(2)]
    main = torch.cuda.current_stream()
    side = torch.cuda.Stream(device=dev)
    stepped = [torch.cuda.Event() for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    for ev in copied:
        ev.record(main)

    def e2e_step(i):
        k = i % 2
        main.wait_event(copied[k])                   # the buffers this play() will overwrite have been copied out
        d_act[k].copy_(h_act[i % E], non_blocking=True)
        obs, reward, _ = game.play(d_act[k])
        flags = game.flags
        stepped[k].record(main)
        with torch.cuda.stream(side):
            side.wait_event(stepped[k])
            h_out[k][0].copy_(obs.board, non_blocking=True)
            h_out[k][1].copy_(reward, non_blocking=True)
            h_out[k][2].copy_(flags, non_blocking=True)
            copied[k].record(side)

    for i in range(4):
        e2e_step(i)
    torch.cuda.synchronize()
    barrier()
    sampler.active = True
    t0 = time.perf_counter()
    for i in range(E):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    sampler.active = False
    e2e_s = reduce_max(e2e_s)
    d2h = n * (cells + 4 + 1)
    e2e = {"value": world * n * E / e2e_s, "unit": "env-steps/s", "h2d_bytes_per_step": n,
           "d2h_bytes_per_step": d2h, "steps": E, "d2h_gbs_per_gpu": d2h * E / e2e_s / 1e9, "numa": numa,
           "what": "Engine.play(): pinned-host uint8 actions -> H2D -> cx_step -> D2H of board, reward, flags every step "
                   "(copy-out of step t on a side stream overlaps H2D + kernel of step t+1); bound by the D2H link"}
    del h_act, h_out

    # ---- secondary contract (BASELINE config 5's policy input): board + layered board per env-step ----
    obs_extra = None
    try:
        if args.obs_reps <= 0:
            raise RuntimeError("skipped (--obs-reps 0)")
        To = 16
        del outs
        torch.cuda.empty_cache()
        o_outs = [game.alloc_rollout(To) for _ in range(2)]
        o_lay = [torch.empty((To, n, nat.n_chars, 5, 5), dtype=torch.uint8, device=dev) for _ in range(2)]

        def obs_issue(i):
            game.rollout_observations(actions[i % n_act][:To], o_outs[i % 2], o_lay[i % 2])

        for i in range(3):
            obs_issue(i)
        reps_o = max(args.obs_reps, 40)
        oms = device_time_ms(obs_issue, 2, reps_o) / reps_o
        ob = 1 + 4 + 1 + cells * (1 + nat.n_chars)
        obs_extra = {"kernel": "k_agent_rollout_obs<TRACK=true>", "alg_bytes_per_env_step": ob,
                     "env_steps_per_sec": n * To / (oms * 1e-3), "achieved_gbs": n * To * ob / (oms * 1e-3) / 1e9,
                     "frac_of_measured_peak": n * To * ob / (oms * 1e-3) / 1e9 / peak, "avg_launch_ms": oms,
                     "launches_timed": reps_o,
                     "fused_steps_per_launch": To, "what": "board u8[25] + layered board u8[7,25] + reward + flags"}
        del o_outs, o_lay
    except Exception as exc:                                     # secondary number: never fail the bench line
        obs_extra = {"error": repr(exc)}

    # ---- episode-return statistics: the one collective of the design (not on the step path) ----
    stats = nat.stats_tensor.clone()
    cxdist.all_reduce_stats(stats)
    summary = cxdist.summarize_stats(stats.cpu())

    # ---- the other BASELINE.json configs (rank 0, one GPU's worth each) ----
    configs = None
    if rank == 0 and world == 1 and not args.no_configs:   # one GPU's worth each: reported on the N = 1 line
        del game, nat
        torch.cuda.empty_cache()
        configs = {}
        jobs = [("hello_world_65536", lambda: measure_config("hello", 65536, 32, peak, 100.0, sampler, "k_generic_rollout")),
                ("demo1_65536", lambda: measure_config("demo1", 65536, 32, peak, 100.0, sampler,
                                                       "k_agent_rollout_lane<TRACK=true> (lane = env, 32 envs per warp)")),
                ("demo1_65536_episode_per_launch", lambda: measure_config(
                    "demo1", 65536, EPISODE_LIMIT, peak, 100.0, sampler,
                    "k_agent_rollout_lane<TRACK=true>, one 100-step episode per launch (examples/actor_critic.py:56)")),
                ("demo2_1048576", lambda: measure_config("demo2", 1 << 20, 20, peak, 100.0, sampler,
                                                         "k_agent_rollout<NG=1,GW=2> (64 envs per warp)")),
                ("demo4_1048576", lambda: measure_config("demo4", 1 << 20, 20, peak, 100.0, sampler,
                                                         "k_agent_rollout<NG=1,GW=2> (64 envs per warp)")),
                ("actor_critic_rollout_4096", lambda: measure_actor_critic(peak, 100.0, sampler))]
        for name, job in jobs:
            try:
                configs[name] = job()
            except Exception as exc:                             # a secondary config never costs the headline line
                configs[name] = {"error": repr(exc)}
            torch.cuda.empty_cache()
    clocks = sampler.stop()

    if rank == 0:
        line = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms / total_steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
            "parity_check": parity, "clocks": clocks, "return_stats": summary,
            "observation_contract_kernel": obs_extra, "configs": configs,
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not p_all:
        sys.stderr.write("bench.py: PARITY CHECK FAILED %r\n" % (p_where,))
        sys.exit(3)


def bind_to_gpu_numa_node(local_rank):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers of the
    end-to-end leg are first-touched in that node's memory (no cross-socket hop on the D2H path).  Returns what
    it found; does nothing on boxes that expose no topology (virtualised hosts report numa_node = -1)."""
    info = {"node": None, "bound": False}
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        with open(path) as f:
            node = int(f.read().strip())
        info["node"] = node
        if node < 0:
            return info
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["bound"] = True
            info["cpus"] = len(allowed)
    except Exception as exc:
        info["error"] = repr(exc)
    return info


_JSON_FD = None


def emit(line):
    """The ONE JSON line of the run, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    args = parse_args()
    # stdout carries ONE JSON line.  NCCL prints its banner / INFO lines on stdout when NCCL_DEBUG asks for them;
    # they are the driver's evidence of the communicator, so NCCL_DEBUG is left alone and everything but the JSON
    # line is sent to stderr at the descriptor level instead.
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args)


if __name__ == "__main__":
    main()
