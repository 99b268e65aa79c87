"""Times the episode statistics (episode_stats=True, CZ_STEP_EPISODE_STATS) against the same steps without them, the two
variants alternating in one process.

    python profiles/microbench/stats_time.py [--out FILE]

1. The in-place step of 131072 two-agent coop_test environments (auto-reset, max_steps 25, fixed device actions) as a
   CUDA graph of 20 steps: dynamics + row writer, and with statistics one cz_stats_kernel more per step.
2. BASELINE config 3: 4096 environments, step_k(64) with device random actions: one launch of the warp kernel
   (cz_warp_kernel<2, G, false> against <2, G, true>).
3. The pipelined step of 131072 environments, 200 steps timed with CUDA events (host-launched: not capturable).
Prints the card's name and power limit with the numbers.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.getcwd())
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from cooking_zoo_b200 import BatchedCookingEnv  # noqa: E402
from grid_time import card, graphed_step, time_graph  # noqa: E402

R2 = ["TomatoLettuceSalad", "CarrotBanana"]


def make(n, stats, max_steps=25, **kw):
    return BatchedCookingEnv(n, "coop_test", "example", 2, max_steps, R2, action_scheme="scheme3", auto_reset=True, seed=1,
                             episode_stats=stats, **kw)


def events(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps


def summary(times):
    off, on = min(times["off"]), min(times["on"])
    return dict(us_off=times["off"], us_on=times["on"], best_off=off, best_on=on, overhead=round(on / off - 1.0, 4))


def in_place(n=131072, rounds=5):
    g = torch.Generator().manual_seed(0)
    actions = [torch.randint(0, 5, (n, 2), generator=g, dtype=torch.uint8).cuda() for _ in range(4)]
    envs = {k: make(n, k == "on") for k in ("off", "on")}
    graphs = {k: graphed_step(e, actions) for k, e in envs.items()}
    times = {k: [] for k in envs}
    for _ in range(rounds):
        for k in envs:
            times[k].append(round(time_graph(graphs[k]), 2))
    fin = int(envs["on"].episode_stats()["finished"].sum())
    for e in envs.values():
        e.close()
    out = dict(summary(times), episodes_finished=fin)
    print(json.dumps({"in_place_131072_graph_of_20": out}), flush=True)
    return out


def config3(n=4096, k=64, rounds=5):
    envs = {key: make(n, key == "on", max_steps=100) for key in ("off", "on")}
    for e in envs.values():
        e.reset()
        for _ in range(3):
            e.step_k(k)
    torch.cuda.synchronize()
    times = {key: [] for key in envs}
    for _ in range(rounds):
        for key, e in envs.items():
            times[key].append(round(events(lambda: e.step_k(k), 10) / k, 3))
    for e in envs.values():
        e.close()
    out = summary(times)
    print(json.dumps({"config3_4096_step_k64_us_per_step": out}), flush=True)
    return out


def pipelined(n=131072, rounds=5, steps=200):
    envs = {key: make(n, key == "on", pipelined=True) for key in ("off", "on")}
    acts = {}
    for key, e in envs.items():
        e.reset()
        acts[key] = e.random_actions(0).clone()
        for _ in range(10):
            e.step(acts[key])
        e.wait()
    torch.cuda.synchronize()
    times = {key: [] for key in envs}

    def run(e, a):
        for _ in range(steps):
            e.step(a)
        e.wait()
    for _ in range(rounds):
        for key, e in envs.items():
            times[key].append(round(events(lambda: run(e, acts[key]), 1) / steps, 2))
    for e in envs.values():
        e.close()
    out = summary(times)
    print(json.dumps({"pipelined_131072_us_per_step": out}), flush=True)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stats_time.py needs a CUDA device")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}), flush=True)
    res = {"card": name, "power_limit": power, "in_place": in_place(), "config3": config3(), "pipelined": pipelined()}
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)
