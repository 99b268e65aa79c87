"""GPU: observations of chosen agents (obs_agents, cz_observe_agents / cz_observe_grid_agents).

The rule (include/cz_b200.h): observation j of every environment is, bit for bit, the one agent obs_agents[j] gets when every
agent's observations are written.  Section 1 holds every path and every subset to a full-row twin with the same seed, section 2
holds the rows to the golden traces and the compiled oracle, section 3 covers a learner beside a device cook, sections 4 and 5
the launches, the full-size batch and CUDA graphs, section 6 the errors."""
import ctypes as C
import itertools
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle.cz_oracle import SpawnStream
from oracle.cz_oracle_c import COracleEnv
from tests.kitchens import kitchen, kitchen_config, plan_class
from tests.replay import golden_files, load_golden, package_recipes
from tests.test_gpu_random_kitchens import N, _make

pytestmark = pytest.mark.gpu
RECIPES = ["TomatoLettuceSalad", "CarrotBanana"]


def _same(a, b, ctx):
    if a.dtype.is_floating_point:
        w = torch.int32 if a.element_size() == 4 else torch.int64
        a, b = a.contiguous().view(w), b.contiguous().view(w)
    assert a.shape == b.shape and torch.equal(a, b), ctx


def _subsets(A):
    return [list(c) for m in range(1, A + 1) for c in itertools.combinations(range(A), m)]


# ---------------------------------------------------------------------------------------------------- 1. every path
# packed plans with <= 32 pairs (A = 1..4), 33-64 pairs (A = 2..4), generic plans with even and odd L (A = 2..4); 1003, 20
# and 12 despawn / respawn agents.  9 (L = 299) and 2 (L = 377) give keep-all blocks of odd N * M * L in float64, 68
# (L = 214) blocks of N * M * L not a multiple of 4 in float32
PATH_KITCHENS = [32, 1017, 1002, 1003, 28, 68, 1011, 13, 20, 9, 12, 2]
SUB_ARMS = {   # name: (environment variables, constructor arguments); N = 3001 is a warp-kernel size for the default arm
    "f64": ({}, {}),
    "lane": ({"CZ_WARP_MAX_ENVS": "0", "CZ_WARP_K_MAX_ENVS": "0"}, {}),
    "generic2": ({"CZ_GENERIC": "2"}, {}),
    "generic1": ({"CZ_GENERIC": "1"}, {}),
    "f32": ({}, {"obs_dtype": torch.float32}),
    "grid": ({}, {"grid": True}),
}
# (kind, steps): single steps, step_k(8) and step_k(8, keep_all=True); auto-reset every 11 steps
OPS = [("step", 1), ("step", 1), ("k", 8), ("step", 1), ("keep", 8), ("step", 1), ("step", 1)]


@pytest.mark.parametrize("seed", PATH_KITCHENS)
def test_every_path_and_subset_equals_the_full_rows(seed, monkeypatch, tmp_path):
    lp, mp, _ = kitchen(seed, str(tmp_path))
    cfg = kitchen_config(seed)
    A = cfg["A"]
    rng = np.random.default_rng(seed)
    acts = torch.from_numpy(rng.integers(0, 8 if cfg["scheme"] == "scheme1" else 5,
                                         size=(sum(k for _, k in OPS), N, A)).astype(np.uint8)).cuda()
    for arm, (env_vars, kw) in SUB_ARMS.items():
        kw = dict(kw)
        if kw.pop("grid", False):
            kw["obs_spaces"] = ["grid"] * A
        common = dict(max_steps=11, auto_reset=True, **kw)
        twin = _make(lp, mp, cfg, seed, N, monkeypatch, env_vars, **common)
        cls = plan_class(twin.tables)
        if arm.startswith("generic") and not cls.startswith("packed"):
            twin.close()
            continue
        subs = {tuple(s): _make(lp, mp, cfg, seed, N, monkeypatch, env_vars, obs_agents=s, **common) for s in _subsets(A)}
        for s, env in subs.items():
            assert env.obs_agents == s and env.obs.shape[1] == len(s)
        want = twin.reset()
        for s, env in subs.items():
            _same(env.reset(), want[:, list(s)], f"kitchen {seed} ({cls}) {arm} {s} reset")
        s0 = 0
        for kind, k in OPS:
            a = acts[s0:s0 + k]
            if kind == "step":
                tw = twin.step(a[0])
            else:
                tw = twin.step_k(k, actions=a, keep_all=kind == "keep")
            tw = [x.clone() for x in tw[:4]]
            for s, env in subs.items():
                ctx = f"kitchen {seed} ({cls}, A={A}) arm {arm} subset {s} {kind} at step {s0}"
                out = env.step(a[0]) if kind == "step" else env.step_k(k, actions=a, keep_all=kind == "keep")
                sel = list(s)
                _same(out[0], tw[0][:, :, sel] if kind == "keep" else tw[0][:, sel], ctx)
                for x, y in zip(out[1:4], tw[1:4]):
                    _same(x, y, ctx)
                _same(env.state, twin.state, ctx)
                _same(env.error_flags, twin.error_flags, ctx)
                if kind != "keep":
                    _same(env.observe(), twin.observe()[:, sel], ctx + " observe()")
            s0 += k
        # episodes ended and restarted (auto-reset) inside the run
        ep = twin.state[twin.tables.num_dyn_slots + A + 5]
        assert int(ep.min()) >= 2, (seed, arm)
        for env in list(subs.values()) + [twin]:
            env.close()


# ---------------------------------------------------------------------------------------------------- 2. oracles
@pytest.mark.parametrize("path", golden_files(), ids=lambda p: p.split("/")[-1][:-4])
def test_one_observer_subsets_replay_golden(path):
    """every one-agent subset of every golden trace: the rows equal the recorded rows of that agent, bit for bit"""
    from cooking_zoo_b200 import BatchedCookingEnv
    g = load_golden(path)
    cfg = g["config"]
    n, A = len(g["layouts"]), cfg["num_agents"]
    kw = {}
    sp = cfg.get("spawn")
    if sp:
        kw = dict(agent_respawn_rate=sp["respawn"], agent_despawn_rate=sp["despawn"], grace_period=sp["grace"], seed=sp["seed"])
    with package_recipes(cfg):
        envs = [BatchedCookingEnv(n, cfg["level"], cfg["meta_file"], A, cfg["max_steps"], cfg["recipes"],
                                  end_condition_all_dishes=cfg["end_all"], reward_scheme=cfg["reward_scheme"],
                                  action_scheme=cfg.get("action_scheme", "scheme3"), layouts=g["layouts"], obs_agents=[i], **kw)
                for i in range(A)]
    want = g["obs"].view(np.uint64)
    for i, env in enumerate(envs):
        got = env.reset(layout_ids=np.arange(n)).cpu().numpy().view(np.uint64)
        assert np.array_equal(got[:, 0], want[:, 0, i]), f"{path} agent {i} reset"
    for t in range(g["actions"].shape[1]):
        live = [k for k in range(n) if t < g["length"][k]]
        if not live:
            break
        for i, env in enumerate(envs):
            for k in live:
                for j in range(A):
                    if g["teleport"][k, t, j, 0] >= 0:
                        env.teleport(k, j, *map(int, g["teleport"][k, t, j]))
            got = env.step(torch.from_numpy(g["actions"][:, t].astype(np.uint8)))[0].cpu().numpy().view(np.uint64)
            for k in live:
                assert np.array_equal(got[k, 0], want[k, t + 1, i]), f"{path} trace {k} agent {i} step {t}"
    for env in envs:
        env.close()


ORACLE_KITCHENS = [1003, 68, 12, 2, 29]
ORACLE_N, ORACLE_STEPS = 256, 40


@pytest.mark.parametrize("seed", ORACLE_KITCHENS)
def test_random_kitchens_against_the_compiled_oracle(seed, monkeypatch, tmp_path):
    lp, mp, _ = kitchen(seed, str(tmp_path))
    cfg = kitchen_config(seed)
    A = cfg["A"]
    sel = [A - 1] if A == 1 else list(range(1, A, 2))
    env = _make(lp, mp, cfg, seed, ORACLE_N, monkeypatch, {}, max_steps=200, obs_agents=sel)
    t = env.tables
    rng = np.random.default_rng(seed)
    lids = rng.integers(0, t.num_layouts, size=ORACLE_N).astype(np.int32)
    oracles = []
    for k in range(ORACLE_N):
        kw = dict(cfg["spawn"], spawn_stream=SpawnStream(seed, k, 1)) if cfg["spawn"] else {}
        oracles.append(COracleEnv(t.layouts[lids[k]], list(cfg["recipes"]), 200, end_condition_all_dishes=cfg["end_all"],
                                  action_scheme=cfg["scheme"], **kw))
    obs = env.reset(layout_ids=lids).cpu().numpy()
    for k in range(ORACLE_N):
        rows = np.stack([oracles[k].observe(i) for i in sel])
        assert np.array_equal(rows.view(np.uint64), obs[k].view(np.uint64)), f"kitchen {seed} env {k} reset"
    alive = set(range(ORACLE_N))
    for s in range(ORACLE_STEPS):
        acts = rng.integers(0, t.num_actions, size=(ORACLE_N, A)).astype(np.uint8)
        obs, rew, term, _, _ = env.step(torch.from_numpy(acts))
        obs, rew, term = obs.cpu().numpy(), rew.cpu().numpy(), term.cpu().numpy()
        for k in sorted(alive):
            ctx = f"kitchen {seed} env {k} step {s}"
            r, te, _, _ = oracles[k].step(acts[k])
            assert np.array_equal(np.asarray(r, np.float64).view(np.uint64), rew[k].view(np.uint64)), ctx
            rows = np.stack([oracles[k].observe(i) for i in sel])
            assert np.array_equal(rows.view(np.uint64), obs[k].view(np.uint64)), ctx
            if any(te):
                alive.discard(k)
    env.close()


# ---------------------------------------------------------------------------------------------------- 3. learner + cook
def _coop(n, **kw):
    from cooking_zoo_b200 import BatchedCookingEnv
    return BatchedCookingEnv(n, "coop_test", "example", 2, kw.pop("max_steps", 20), RECIPES, action_scheme="scheme3",
                             auto_reset=True, seed=11, **kw)


@pytest.mark.parametrize("stats", [False, True])
def test_learner_beside_a_cook(stats):
    """cook_agents=[1], obs_agents=[0] against cook_agents=[1] with every row: single steps and step_k(64), which stays one
    warp-kernel launch plus one subset write"""
    n = 4096
    env, twin = _coop(n, cook_agents=[1], obs_agents=[0], episode_stats=stats), _coop(n, cook_agents=[1], episode_stats=stats)
    assert env.obs.shape == (n, 1, env.obs_len)
    _same(env.reset(), twin.reset()[:, [0]], "reset")
    a = torch.zeros((n, 2), dtype=torch.uint8, device="cuda")
    for s in range(30):
        a = env.random_actions(s).clone()
        o, r, te, tu, _ = env.step(a)
        to, tr, tte, ttu, _ = twin.step(a)
        for x, y in ((o, to[:, [0]]), (r, tr), (te, tte), (tu, ttu), (env.actions_taken, twin.actions_taken),
                     (env.cook_step_crashed, twin.cook_step_crashed), (env.state, twin.state)):
            _same(x, y, f"step {s}")
    l0 = env.lib.cz_launch_count()
    o = env.step_k(64, action_step=30)[0]
    assert env.lib.cz_launch_count() - l0 == 2
    to = twin.step_k(64, action_step=30)[0]
    _same(o, to[:, [0]], "step_k(64)")
    _same(env.state, twin.state, "step_k(64) state")
    _same(env.actions_taken, twin.actions_taken, "step_k(64) actions_taken")
    _same(env.cook_step_crashed, twin.cook_step_crashed, "step_k(64) crashed")
    assert int(env.state[env.tables.num_dyn_slots + 2 + 5].min()) >= 3       # EPISODE row: auto-resets inside the launch
    if stats:
        a_, b_ = env.episode_stats(), twin.episode_stats()
        for k in a_:
            _same(a_[k], b_[k], k)
    env.close(); twin.close()


# ---------------------------------------------------------------------------------------------------- 4. launches
_PROFILE = r"""
import json, os, sys
import torch
sys.path.insert(0, sys.argv[1])
from cooking_zoo_b200 import BatchedCookingEnv
out = {}
for name, n, kw, k in [("warp", 2048, {}, 1), ("k8", 2048, {}, 8), ("two", 32768, {}, 1), ("f32", 32768, {"obs_dtype": torch.float32}, 1),
                       ("grid", 32768, {"obs_spaces": ["grid"] * 2}, 1)]:
    for sel in ("none", "all", "one"):
        env = BatchedCookingEnv(n, "coop_test", "example", 2, 25, ["TomatoLettuceSalad", "CarrotBanana"], action_scheme="scheme3",
                                auto_reset=True, obs_agents={"none": None, "all": [0, 1], "one": [0]}[sel], **kw)
        env.reset()
        a = env.random_actions(0)
        go = (lambda: env.step_k(k)) if k > 1 else (lambda: env.step(a))
        go(); torch.cuda.synchronize()
        l0 = env.lib.cz_launch_count()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            go()
            torch.cuda.synchronize()
        names = sorted({e.key[e.key.index("cz_"):].split("(")[0] for e in prof.key_averages() if "cz_" in e.key})
        out[name + "_" + sel] = {"launches": env.lib.cz_launch_count() - l0, "kernels": names}
        env.close()
print(json.dumps(out))
"""


def test_launches_and_kernels():
    """obs_agents=None and obs_agents naming every agent launch the same kernels; a subset runs the dynamics without rows
    (the warp kernel for small batches and K steps, the dynamics-only kernel for large ones) and one subset writer"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", _PROFILE, root], cwd=root, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    print(out)
    writer = {"warp": "cz_obs_agents_kernel<double, 2, false, 2>", "k8": "cz_obs_agents_kernel<double, 2, false, 2>",
              "two": "cz_obs_agents_kernel<double, 2, false, 2>", "f32": "cz_obs_agents_kernel<float, 2, false, 2>",
              "grid": "cz_grid_agents_kernel<2>"}
    for name, w in writer.items():
        none, full, one = out[name + "_none"], out[name + "_all"], out[name + "_one"]
        assert none == full, (name, none, full)
        assert one["launches"] == 2, (name, one)
        if name in ("warp", "k8"):
            assert one["kernels"] == sorted(["cz_warp_kernel<2, 16, false, false>", w]), (name, one)
        else:
            assert w in one["kernels"] and any(k.startswith("cz_env_kernel<0, 2, 2>") for k in one["kernels"]), (name, one)
        assert not any(k.startswith(("cz_obs_agents", "cz_grid_agents")) for k in none["kernels"]), (name, none)


# ---------------------------------------------------------------------------------------------------- 5. scale, graphs
@pytest.mark.parametrize("mode", ["f64", "f32", "grid"])
def test_full_scale_in_place_with_masked_resets(mode):
    n = 131072
    kw = {"f64": {}, "f32": {"obs_dtype": torch.float32}, "grid": {"obs_spaces": ["grid"] * 2}}[mode]
    env, twin = _coop(n, obs_agents=[1], max_steps=15, **kw), _coop(n, max_steps=15, **kw)
    _same(env.reset(), twin.reset()[:, [1]], "reset")
    reset_mask = torch.from_numpy(np.arange(n) % 3 == 0)
    for s in range(20):
        if s == 9:
            lids = twin.default_layout_ids(episode=5)
            _same(env.reset(layout_ids=lids, mask=reset_mask), twin.reset(layout_ids=lids, mask=reset_mask)[:, [1]], "masked")
        a = twin.random_actions(s).clone()
        o = env.step(a)
        t = twin.step(a)
        ctx = f"{mode} step {s}"
        _same(o[0], t[0][:, [1]], ctx)
        for x, y in zip(o[1:4], t[1:4]):
            _same(x, y, ctx)
        _same(env.state, twin.state, ctx); _same(env.error_flags, twin.error_flags, ctx)
    env.close(); twin.close()


@pytest.mark.parametrize("n", [2048, 20000])
def test_cuda_graph_equals_eager(n):
    def run(graph):
        env = _coop(n, cook_agents=[1], obs_agents=[0], max_steps=6)
        env.reset()
        a = env.random_actions(0)
        if graph:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                env.step(a)                                  # warm-up outside the capture
            torch.cuda.current_stream().wait_stream(s)
            env.reset()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for _ in range(20):
                    env.step(a)
            g.replay()
        else:
            env.step(a)
            env.reset()
            for _ in range(20):
                env.step(a)
        torch.cuda.synchronize()
        out = {"state": env.state.clone(), "obs": env.obs.clone(), "reward": env.reward.clone()}
        env.close()
        return out
    eager, graph = run(False), run(True)
    for k in eager:
        _same(eager[k], graph[k], k)


# ---------------------------------------------------------------------------------------------------- 6. errors
def test_errors():
    from cooking_zoo_b200 import _native, MixedAgentCookingEnv
    from cooking_zoo_b200.wrappers import ParallelCookingEnv
    env = _coop(64, obs_agents=[0])
    lib, h = env.lib, env._handle
    env.reset()
    st = env.state.data_ptr()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rows = torch.zeros(64 * 2 * env.obs_len + 2, dtype=torch.float64, device="cuda")
    grid = torch.zeros(64 * 2 * len(env.grid_channels) * env.tables.width * env.tables.height + 16, dtype=torch.uint8,
                       device="cuda")
    o, g = rows.data_ptr(), grid.data_ptr()
    for mask, rc in ((0, -1), (4, -1), (1 << 31, -1), (3, 0), (1, 0), (2, 0)):
        assert lib.cz_observe_agents(h, st, mask, o, 0, 64, s) == rc, mask
        assert lib.cz_observe_grid_agents(h, st, mask, g, 64, s) == rc, mask
    assert lib.cz_observe_agents(h, st, 0, o, 0, 64, s) == -1 and b"agent_mask" in lib.cz_last_error()
    assert lib.cz_observe_agents(None, st, 1, o, 0, 64, s) == -1
    assert lib.cz_observe_agents(h, None, 1, o, 0, 64, s) == -1
    assert lib.cz_observe_agents(h, st, 1, None, 0, 64, s) == -1
    assert lib.cz_observe_agents(h, st, 1, o, _native.STEP_AUTO_RESET, 64, s) == -1        # a flag other than OBS_F32
    assert lib.cz_observe_agents(h, st, 1, o + 4, 0, 64, s) == -1                          # float64 rows at a 4-byte offset
    assert lib.cz_observe_agents(h, st, 1, o + 2, _native.STEP_OBS_F32, 64, s) == -1       # float32 rows at a 2-byte offset
    assert lib.cz_observe_agents(h, st, 1, o + 8, 0, 64, s) == 0                           # 8-byte aligned float64 rows work
    assert lib.cz_observe_agents(h, st, 1, o + 4, _native.STEP_OBS_F32, 64, s) == 0
    assert lib.cz_observe_grid_agents(None, st, 1, g, 64, s) == -1
    assert lib.cz_observe_grid_agents(h, None, 1, g, 64, s) == -1
    assert lib.cz_observe_grid_agents(h, st, 1, None, 64, s) == -1
    assert lib.cz_observe_agents(h, st, 1, o, 0, 0, s) == 0 and lib.cz_observe_grid_agents(h, st, 1, g, 0, s) == 0
    # the grid at an odd byte offset: the same bytes as at an aligned one
    torch.cuda.synchronize()
    E = len(env.grid_channels) * env.tables.width * env.tables.height
    assert lib.cz_observe_grid_agents(h, st, 2, g + 3, 64, s) == 0
    torch.cuda.synchronize()
    odd = grid[3:3 + 64 * E].clone()
    assert lib.cz_observe_grid_agents(h, st, 2, g, 64, s) == 0
    torch.cuda.synchronize()
    assert torch.equal(odd, grid[:64 * E])
    full = env.grid_observation()
    assert torch.equal(odd.view(64, E), full[:, 1].reshape(64, E))
    for bad in ([], [0, 0], [2], [-1], [1, 0]):
        with pytest.raises(ValueError):
            _coop(64, obs_agents=bad)
    with pytest.raises(NotImplementedError):
        _coop(64, obs_agents=[0], pipelined=True)
    _coop(64, obs_agents=[0, 1], pipelined=True).close()                                 # every agent: today's path
    with pytest.raises(NotImplementedError):
        MixedAgentCookingEnv([1, 2, 2], "coop_test", "example", 20, RECIPES, action_scheme="scheme3", obs_agents=[0])
    with pytest.raises(NotImplementedError):
        ParallelCookingEnv("coop_test", "example", 2, 20, RECIPES, action_scheme="scheme3", obs_agents=[0])
    assert _coop(64).obs_agents == (0, 1)
    env.close()
