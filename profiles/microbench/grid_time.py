"""Times the grid observation (cz_observe_grid): the writer alone, and the in-place grid step against the feature-vector
steps in the same process.

    python profiles/microbench/grid_time.py [--out FILE]

1. The writer alone on a stepped state, CUDA events around 50 launches: 131072 two-agent coop_test environments, and the
   open 4-agent kitchen (tests/golden/levels/open4.json) with 1-4 agents at 65536 environments.  Bytes = grid bytes written
   + state bytes read; the fraction is of 6550 GB/s (the write rate the project measured as its ceiling, DESIGN section 4).
2. The in-place step of 131072 coop_test environments (auto-reset, fixed device actions) as a CUDA graph of 20 steps, in
   grid mode and with float64 / float32 feature-vector rows, alternating the three for three rounds.
Prints the card's name and power limit with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.getcwd())
from cooking_zoo_b200 import BatchedCookingEnv  # noqa: E402

R2 = ["TomatoLettuceSalad", "CarrotBanana"]
R4 = ["TomatoLettuceSalad", "CarrotBanana", "TomatoSalad", "no_recipe"]
CEILING_GBS = 6550.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as ex:      # the number is still reported, without the power limit
        power = f"unknown ({ex!r})"
    return name, power


def make(n, agents=2, open4=False, **kw):
    if open4:
        return BatchedCookingEnv(n, "tests/golden/levels/open4.json", "tests/golden/levels/meta4.json", agents, 400, R4[:agents],
                                 end_condition_all_dishes=True, action_scheme="scheme3", layout_pool_size=64, auto_reset=True,
                                 seed=1, **kw)
    return BatchedCookingEnv(n, "coop_test", "example", agents, 400, R2[:agents], end_condition_all_dishes=True,
                             action_scheme="scheme3", layout_pool_size="auto", auto_reset=True, seed=1, **kw)


def writer_alone(n, agents=2, open4=False):
    env = make(n, agents, open4, obs_spaces=["grid"] * agents)
    env.reset()
    for s in range(8):
        env.step(env.random_actions(s))
    for _ in range(5):
        env.observe()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        env.observe()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / 50
    written = env.obs.numel()
    read = env.state.numel() * 4
    gbs = (written + read) / us / 1e3
    out = dict(kitchen="open4" if open4 else "coop_test", agents=agents, envs=n, channels=len(env.grid_channels),
               bytes_per_env=written // n, us=round(us, 2), grid_bytes=written, state_bytes=read, tb_s=round(gbs / 1e3, 3),
               fraction_of_6550=round(gbs / CEILING_GBS, 3))
    print(json.dumps(out), flush=True)
    env.close()
    return out


def graphed_step(env, actions, steps=20):
    env.reset()
    for s in range(3):
        env.step(actions[s % len(actions)])
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
            for s in range(steps):
                env.step(actions[s % len(actions)])
    torch.cuda.current_stream().wait_stream(side)
    graph.replay()
    torch.cuda.synchronize()
    return graph


def time_graph(graph, steps=20, replays=10):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    graph.replay()
    e0.record()
    for _ in range(replays):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (replays * steps)


def step_comparison(n=131072, rounds=3):
    g = torch.Generator().manual_seed(0)
    actions = [torch.randint(0, 5, (n, 2), generator=g, dtype=torch.uint8).cuda() for _ in range(4)]
    envs = {"grid": make(n, obs_spaces=["grid"] * 2), "f64": make(n), "f32": make(n, obs_dtype=torch.float32)}
    graphs = {k: graphed_step(e, actions) for k, e in envs.items()}
    times = {k: [] for k in envs}
    for r in range(rounds):
        for k in envs:
            times[k].append(round(time_graph(graphs[k]), 2))
    out = {}
    for k, e in envs.items():
        nbytes = e.obs.numel() * e.obs.element_size()
        best = min(times[k])
        out[k] = dict(us_per_step=times[k], obs_bytes=nbytes, obs_tb_s_best=round(nbytes / best / 1e6, 3))
    print(json.dumps({"in_place_step_131072_coop_test_graph_of_20": out}), flush=True)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("grid_time.py needs a CUDA device")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}), flush=True)
    res = {"card": name, "power_limit": power, "writer": [writer_alone(131072)]}
    for a in (1, 2, 3, 4):
        res["writer"].append(writer_alone(65536, a, open4=True))
    res["step"] = step_comparison()
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)
