"""Times cook agents (cook_agents=..., CZ_STEP_COOK_AGENTS) against the other ways to run the same closed loop, the arms
alternating in one process.

    python profiles/microbench/cook_agents_time.py [--out FILE]

1. 4096 two-agent coop_test environments, both agents cooks (auto-reset, max_steps 100), microseconds per step:
   - "fused": step_k(64), one launch of cz_warp_kernel<2, G, true, false>;
   - "fallback": the same call with CZ_WARP_K_MAX_ENVS=0, the library's per-step loop (64 x (merge kernel + step));
   - "compose_graph": a CUDA graph of 64 x (heuristic_actions + torch merge + step) on an environment without cook agents.
2. 131072 environments, agent 0 a cook and agent 1 a learner with fixed actions, microseconds per step:
   - in place, CUDA graphs of 20 steps: "partner" (step with cook_agents=[0]) against "compose" (heuristic_actions +
     torch.where + step);
   - pipelined, 200 host-launched steps timed with CUDA events: the same two arms.
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
from grid_time import card  # noqa: E402

R2 = ["TomatoLettuceSalad", "CarrotBanana"]


def make(n, max_steps=100, env_vars=None, **kw):
    os.environ.update(env_vars or {})
    try:
        return BatchedCookingEnv(n, "coop_test", "example", 2, max_steps, R2, action_scheme="scheme3", auto_reset=True, seed=1,
                                 **kw)
    finally:
        for k in env_vars or {}:
            del os.environ[k]


def events(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps


def capture(fn):
    """CUDA graph of fn() (warmed up once outside the capture)"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    graph.replay()
    torch.cuda.synchronize()
    return graph


def compose_step(env, mask, a):
    cook, _ = env.heuristic_actions()
    env.step(torch.where(mask, cook, a))


def closed_loop(n=4096, k=64, rounds=5):
    both = [0, 1]
    envs = {"fused": make(n, cook_agents=both), "fallback": make(n, cook_agents=both, env_vars={"CZ_WARP_K_MAX_ENVS": "0"}),
            "compose": make(n)}
    zeros = torch.zeros((n, 2), dtype=torch.uint8, device="cuda")
    mask = torch.ones((n, 2), dtype=torch.bool, device="cuda")
    for e in envs.values():
        e.reset()
    runs = {"fused": lambda: envs["fused"].step_k(k), "fallback": lambda: envs["fallback"].step_k(k)}
    g = capture(lambda: [compose_step(envs["compose"], mask, zeros) for _ in range(k)])
    runs["compose_graph"] = g.replay
    for f in runs.values():
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    times = {key: [] for key in runs}
    for _ in range(rounds):
        for key, f in runs.items():
            times[key].append(round(events(f, 10) / k, 3))
    for e in envs.values():
        e.close()
    out = {key: dict(us_per_step=v, best=min(v)) for key, v in times.items()}
    print(json.dumps({"closed_loop_4096_k64_us_per_step": out}), flush=True)
    return out


def partner(n=131072, steps=20, rounds=5):
    mask = torch.zeros((n, 2), dtype=torch.bool, device="cuda")
    mask[:, 0] = True
    a = torch.randint(0, 5, (n, 2), generator=torch.Generator().manual_seed(0), dtype=torch.uint8).cuda()
    out = {}
    # in place: CUDA graphs of `steps` steps
    envs = {"partner": make(n, cook_agents=[0]), "compose": make(n)}
    for e in envs.values():
        e.reset()
    graphs = {"partner": capture(lambda: [envs["partner"].step(a) for _ in range(steps)]),
              "compose": capture(lambda: [compose_step(envs["compose"], mask, a) for _ in range(steps)])}
    times = {key: [] for key in graphs}
    for _ in range(rounds):
        for key, g in graphs.items():
            times[key].append(round(events(g.replay, 10) / steps, 2))
    for e in envs.values():
        e.close()
    out["in_place_graph"] = {key: dict(us_per_step=v, best=min(v)) for key, v in times.items()}
    # pipelined: host-launched steps
    envs = {"partner": make(n, cook_agents=[0], pipelined=True), "compose": make(n, pipelined=True)}
    runs = {"partner": lambda: envs["partner"].step(a), "compose": lambda: compose_step(envs["compose"], mask, a)}

    def run(key, reps):
        for _ in range(reps):
            runs[key]()
        envs[key].wait()
    for key, e in envs.items():
        e.reset()
        run(key, 10)
    torch.cuda.synchronize()
    times = {key: [] for key in runs}
    for _ in range(rounds):
        for key in runs:
            times[key].append(round(events(lambda: run(key, 200), 1) / 200, 2))
    for e in envs.values():
        e.close()
    out["pipelined_events"] = {key: dict(us_per_step=v, best=min(v)) for key, v in times.items()}
    print(json.dumps({"partner_131072_us_per_step": out}), flush=True)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cook_agents_time.py needs a CUDA device")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}), flush=True)
    res = {"card": name, "power_limit": power, "closed_loop": closed_loop(), "partner": partner()}
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)
