"""Times observations of chosen agents (obs_agents=..., cz_observe_agents / cz_observe_grid_agents) against every agent's
observations, the arms alternating in one process.  131072 two-agent coop_test environments with auto-reset.

    python profiles/microbench/obs_agents_time.py [--out FILE]

1. The writers alone, on a fixed state (CUDA events over 50 calls): the full-row writer (observe()) against the subset
   writer of agent 0, in float64, float32 and grid mode; microseconds per call and TB/s over the bytes of the output
   (computed from its shape: the writers are write streams, their reads hit L2).
2. The in-place step under CUDA graphs of 20 steps, microseconds per step: full observations against obs_agents=[0], in
   float64, float32 and grid mode.
3. The same for a learner beside a device cook: cook_agents=[1], obs_agents=[0] against cook_agents=[1] alone.
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
from cook_agents_time import capture, events  # noqa: E402

R2 = ["TomatoLettuceSalad", "CarrotBanana"]
N = 131072
MODES = {"f64": {}, "f32": {"obs_dtype": torch.float32}, "grid": {"obs_spaces": ["grid"] * 2}}


def make(**kw):
    return BatchedCookingEnv(N, "coop_test", "example", 2, 100, R2, action_scheme="scheme3", auto_reset=True, seed=1, **kw)


def alternate(runs, reps, per, rounds):
    """runs: name -> callable; `rounds` passes over the arms in turn, each timing `reps` calls; microseconds per `per`"""
    for f in runs.values():
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    times = {key: [] for key in runs}
    for _ in range(rounds):
        for key, f in runs.items():
            times[key].append(round(events(f, reps) / per, 2))
    return {key: dict(us=v, best=min(v)) for key, v in times.items()}


def writers(rounds=5):
    out = {}
    for mode, kw in MODES.items():
        envs = {"full": make(**kw), "obs_agents_0": make(obs_agents=[0], **kw)}
        for e in envs.values():
            e.reset()
        res = alternate({key: e.observe for key, e in envs.items()}, 50, 1, rounds)
        for key, e in envs.items():
            nbytes = e.obs.numel() * e.obs.element_size()
            res[key]["bytes"] = nbytes
            res[key]["tb_per_s_best"] = round(nbytes / (res[key]["best"] * 1e-6) / 1e12, 2)
            e.close()
        out[mode] = res
        print(json.dumps({"writer_alone_" + mode: res}), flush=True)
    return out


def steps(arms, rounds=5, n_steps=20):
    """arms: name -> constructor arguments; CUDA graphs of n_steps in-place steps on fixed random actions"""
    a = torch.randint(0, 5, (N, 2), generator=torch.Generator().manual_seed(0), dtype=torch.uint8).cuda()
    envs = {key: make(**kw) for key, kw in arms.items()}
    graphs = {}
    for key, e in envs.items():
        e.reset()
        graphs[key] = capture(lambda e=e: [e.step(a) for _ in range(n_steps)])
    res = alternate({key: g.replay for key, g in graphs.items()}, 10, n_steps, rounds)
    for e in envs.values():
        e.close()
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("obs_agents_time.py needs a CUDA device")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}), flush=True)
    res = {"card": name, "power_limit": power, "writer_alone": writers(), "step_graph_us": {}}
    for mode, kw in MODES.items():
        res["step_graph_us"][mode] = steps({"full": kw, "obs_agents_0": dict(kw, obs_agents=[0])})
        print(json.dumps({"step_graph_" + mode: res["step_graph_us"][mode]}), flush=True)
    res["step_graph_us"]["cook_1"] = steps({"cook_1": {"cook_agents": [1]}, "cook_1_obs_agents_0": {"cook_agents": [1],
                                                                                                    "obs_agents": [0]}})
    print(json.dumps({"step_graph_cook_1": res["step_graph_us"]["cook_1"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)
