"""Development aid (round 2): single-step latency and small/mid-batch throughput of the single-agent kernels.
Usage: python scripts/r02_probe.py [step|obs]..."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from campx_b200.runtime import NativeGame
from tests.expected_specs import expected_spec


def timed(fn, lead, count):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    for i in range(lead): fn(i)
    e0.record()
    for i in range(count): fn(lead + i)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / count


def graph_of(fn, k):
    side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(k): fn(i)
    torch.cuda.current_stream().wait_stream(side); torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(k): fn(i)
    return g


def step_probe():
    for n in (4096, 65536, 1 << 20):
        for flat in ("step_composer", "no_step_composer"):
            os.environ["CX_ROUTE"] = flat
            g = NativeGame(expected_spec("boat_race", max_episode_steps=100, track_returns=True), n)
            nb = max(2, int(300e6 // (n * 31)) + 1)
            bufs = [g.alloc_outputs() for _ in range(nb)]
            acts = g.fill_actions(nb, seed=1)
            gr = graph_of(lambda i: g.step(acts[i % nb], *bufs[i % nb]), nb)
            ms = timed(lambda i: gr.replay(), 1, max(3, int(20 / (nb * 0.01)))) / nb
            print("cx_step n=%d %s: %.2f us/step  %.1f GB/s" % (n, flat, ms * 1e3, n * 31 / ms / 1e6), flush=True)
        os.environ.pop("CX_ROUTE", None)
        for dt in (torch.uint8, torch.float32, torch.bfloat16):
            g = NativeGame(expected_spec("boat_race", max_episode_steps=100, track_returns=True), n)
            es = torch.empty((), dtype=dt).element_size()
            per = 31 + 175 * es
            nb = max(2, int(300e6 // (n * per)) + 1)
            bufs = [g.alloc_outputs() for _ in range(nb)]
            lay = [torch.empty((n, 7, 5, 5), dtype=dt, device="cuda") for _ in range(nb)]
            acts = g.fill_actions(nb, seed=1)
            gr = graph_of(lambda i: g.step_observations(acts[i % nb], bufs[i % nb][0], lay[i % nb], bufs[i % nb][1], bufs[i % nb][2]), nb)
            ms = timed(lambda i: gr.replay(), 1, max(3, int(20 / (nb * 0.01)))) / nb
            print("cx_step_observations n=%d %s: %.2f us/step  %.1f GB/s" % (n, dt, ms * 1e3, n * per / ms / 1e6), flush=True)


def obs_probe():
    T = 16
    for n in (4096, 65536, 1 << 18, 1 << 20):
        g = NativeGame(expected_spec("boat_race", max_episode_steps=100, track_returns=True), n)
        nb = max(2, int(400e6 // (n * T * 206)) + 1)
        bufs = [g.alloc_outputs(T) for _ in range(nb)]
        lay = [torch.empty((T, n, 7, 5, 5), dtype=torch.uint8, device="cuda") for _ in range(nb)]
        acts = [g.fill_actions(T, seed=1, t0=i * T) for i in range(nb)]
        gr = graph_of(lambda i: g.rollout_observations(acts[i % nb], bufs[i % nb][0], lay[i % nb], bufs[i % nb][1], bufs[i % nb][2]), nb)
        ms = timed(lambda i: gr.replay(), 1, max(3, int(30 / (nb * 0.05)))) / nb
        print("obs n=%d T=%d: %.4f ms/launch  %.0f GB/s (%.1f%%)" % (n, T, ms, n * T * 206 / ms / 1e6, n * T * 206 / ms / 1e6 / 65.341), flush=True)
        del g, bufs, lay, acts, gr


if __name__ == "__main__":
    what = sys.argv[1:] or ["step", "obs"]
    if "step" in what: step_probe()
    if "obs" in what: obs_probe()




def tsweep_probe():
    """Steps per launch: Hello World (generic kernel) and mid-size single-agent batches (lockstep / drift effect)."""
    for world, n, Ts in (("hello", 65536, (8, 12, 16, 24, 32)), ("hello", 1 << 18, (8, 12, 16, 24, 32)),
                         ("demo1", 1 << 18, (12, 16, 20, 24, 32)), ("demo1", 65536, (16, 32, 64))):
        for T in Ts:
            g = NativeGame(expected_spec(world, max_episode_steps=100, track_returns=(world != "hello")), n)
            per = (478 if world == "hello" else 31)
            nb = max(2, int(600e6 // (n * T * per)) + 1)
            bufs = [g.alloc_outputs(T) for _ in range(nb)]
            acts = [g.fill_actions(T, seed=543 + i) for i in range(nb)]
            if world == "hello":
                acts = [torch.where(a == 4, torch.zeros_like(a), a).contiguous() for a in acts]   # no quits: steady state
            gr = graph_of(lambda i: g.rollout(acts[i % nb], *bufs[i % nb]), max(nb, 8))
            per_replay = timed(lambda i: gr.replay(), 1, 3)
            timed(lambda i: gr.replay(), 0, max(3, int(100 / per_replay)))            # back under load
            ms = timed(lambda i: gr.replay(), 1, max(6, int(60 / per_replay))) / max(nb, 8)
            state = (942 if world == "hello" else 14)
            alg = n * (T * per + state)
            print("%s n=%d T=%d: %.4f ms/launch  %.3e env-steps/s  %.0f GB/s (%.1f%%)" % (
                world, n, T, ms, n * T / ms * 1e3, alg / ms / 1e6, alg / ms / 1e6 / 65.341), flush=True)
            del g, bufs, acts, gr


if __name__ == "__main__" and "tsweep" in sys.argv[1:]:
    tsweep_probe()


def stg_sweep():
    """Small batches: launch time against steps per launch (slope = per-step time, intercept = fixed cost per launch),
    with and without episode tracking, for the 64-env tile build and the STG lane kernel."""
    for mode, route in (("tile64", "tile64"), ("stg", "lane")):
        os.environ["CX_ROUTE"] = route
        for track in (True, False):
            for n in (4096, 65536):
                for T in (8, 16, 32, 64, 128):
                    kw = dict(max_episode_steps=100, track_returns=True) if track else dict()
                    g = NativeGame(expected_spec("demo1", **kw), n)
                    nb = max(2, int(400e6 // (n * T * 31)) + 1)
                    bufs = [g.alloc_outputs(T) for _ in range(nb)]
                    acts = [g.fill_actions(T, seed=1, t0=i * T) for i in range(nb)]
                    gr = graph_of(lambda i: g.rollout(acts[i % nb], *bufs[i % nb]), nb)
                    ms = timed(lambda i: gr.replay(), 2, max(3, int(30 / (nb * 0.03)))) / nb
                    print("%s track=%d n=%d T=%d: %.2f us/launch  %.3f us/step  %.0f GB/s (%.1f%%)" % (
                        mode, track, n, T, ms * 1e3, ms * 1e3 / T, n * T * 31.44 / ms / 1e6, n * T * 31.44 / ms / 1e6 / 65.341), flush=True)
                    del g, bufs, acts, gr
    os.environ.pop("CX_ROUTE", None)


if __name__ == "__main__":
    if "tsweep" in sys.argv[1:]: tsweep_probe()
    if "stgsweep" in sys.argv[1:]: stg_sweep()


def big_sweep():
    """Large batches: kernel build x steps per launch (boat_race, the bench workload)."""
    for n in (1 << 19, 1 << 20):
        for mode, route in (("tile64", "tile64"), ("tile128", "tile128"), ("tile256", "tile256"), ("stg", "lane")):
            if os.environ.get("PROBE_MODES") and mode not in os.environ["PROBE_MODES"].split(","):
                continue
            for T in (12, 16, 20, 24, 32, 48):
                os.environ["CX_ROUTE"] = route
                g = NativeGame(expected_spec("boat_race", max_episode_steps=100, track_returns=True), n)
                nb = max(2, int(1300e6 // (n * T * 31)) + 1)
                bufs = [g.alloc_outputs(T) for _ in range(nb)]
                acts = [g.fill_actions(T, seed=1, t0=i * T) for i in range(nb)]
                fn = lambda i: g.rollout(acts[i % nb], *bufs[i % nb])
                per = timed(fn, 2, 4)
                timed(fn, 0, max(4, int(100 / per)))
                ms = timed(fn, 2, max(8, int(150 / per)))
                alg = n * (T * 31 + 14)
                print("boat_race n=%d T=%d %s: %.4f ms/launch  %.3e env-steps/s  %.0f GB/s (%.1f%%)" % (
                    n, T, mode, ms, n * T / ms * 1e3, alg / ms / 1e6, alg / ms / 1e6 / 65.341), flush=True)
                del g, bufs, acts
    os.environ.pop("CX_ROUTE", None)


if __name__ == "__main__":
    if "bigsweep" in sys.argv[1:]: big_sweep()


def lane_knobs():
    """k_agent_rollout_lane at BASELINE config 1 (Demo 1, 65,536 envs) by batch size and steps per launch, against the
    routes LANEKNOB_MODES names (auto or CX_ROUTE values, e.g. auto,tile64)."""
    for mode in (os.environ.get("LANEKNOB_MODES", "auto").split(",")):
        os.environ.pop("CX_ROUTE", None)
        if mode != "auto": os.environ["CX_ROUTE"] = mode
        for n in [int(x) for x in os.environ.get("LANEKNOB_SIZES", "4096,16384,32768,65536,131072,262144").split(",")]:
            for T in (32, 100):
                g = NativeGame(expected_spec("demo1", max_episode_steps=100, track_returns=True), n)
                nb = max(2, int(400e6 // (n * T * 31)) + 1)
                bufs = [g.alloc_outputs(T) for _ in range(nb)]
                acts = [g.fill_actions(T, seed=1, t0=i * T) for i in range(nb)]
                gr = graph_of(lambda i: g.rollout(acts[i % nb], *bufs[i % nb]), max(nb, 8))
                per = timed(lambda i: gr.replay(), 1, 3)
                timed(lambda i: gr.replay(), 0, max(3, int(100 / per)))
                ms = timed(lambda i: gr.replay(), 1, max(6, int(60 / per))) / max(nb, 8)
                alg = n * (T * 31 + 14)
                print("lane %s n=%d T=%d: %.2f us/launch  %.0f GB/s (%.1f%%)" % (mode, n, T, ms * 1e3, alg / ms / 1e6, alg / ms / 1e6 / 65.341), flush=True)
                del g, bufs, acts, gr
    os.environ.pop("CX_ROUTE", None)


if __name__ == "__main__":
    if "laneknobs" in sys.argv[1:]: lane_knobs()


def t_small():
    """Large batches, few steps per launch: which tile build?"""
    for n in (1 << 19, 1 << 20):
        for mode in ("tile64", "tile128", "tile256"):   # single steps of these batches skip the step composer
            for T in (1, 2, 4, 8):
                os.environ["CX_ROUTE"] = mode
                g = NativeGame(expected_spec("boat_race", max_episode_steps=100, track_returns=True), n)
                nb = max(2, int(400e6 // (n * T * 31)) + 1)
                bufs = [g.alloc_outputs(T) for _ in range(nb)]
                acts = [g.fill_actions(T, seed=1, t0=i * T) for i in range(nb)]
                gr = graph_of(lambda i: g.rollout(acts[i % nb], *bufs[i % nb]), nb)
                per = timed(lambda i: gr.replay(), 1, 3)
                ms = timed(lambda i: gr.replay(), 1, max(6, int(40 / per))) / nb
                alg = n * (T * 31 + 14)
                print("boat_race n=%d T=%d %s: %.2f us/launch  %.0f GB/s (%.1f%%)" % (n, T, mode, ms * 1e3, alg / ms / 1e6, alg / ms / 1e6 / 65.341), flush=True)
                del g, bufs, acts, gr
    os.environ.pop("CX_ROUTE", None)


if __name__ == "__main__":
    if "tsmall" in sys.argv[1:]: t_small()


def ragged():
    """Batches that are not a whole number of warp tiles: how far off the aligned path are they?"""
    for n in (1 << 19, 500000, 500016, 500001, 65536, 65552, 65521):
        T = 20
        g = NativeGame(expected_spec("boat_race", max_episode_steps=100, track_returns=True), n)
        nb = max(2, int(700e6 // (n * T * 31)) + 1)
        bufs = [g.alloc_outputs(T) for _ in range(nb)]
        acts = [g.fill_actions(T, seed=1, t0=i * T) for i in range(nb)]
        fn = lambda i: g.rollout(acts[i % nb], *bufs[i % nb])
        gr = graph_of(fn, max(nb, 8))
        per = timed(lambda i: gr.replay(), 1, 3)
        ms = timed(lambda i: gr.replay(), 1, max(6, int(60 / per))) / max(nb, 8)
        alg = n * (T * 31 + 14)
        print("ragged n=%d T=%d: %.2f us/launch  %.0f GB/s (%.1f%%)" % (n, T, ms * 1e3, alg / ms / 1e6, alg / ms / 1e6 / 65.341), flush=True)
        del g, bufs, acts, gr


if __name__ == "__main__":
    if "ragged" in sys.argv[1:]: ragged()
