"""GPU: cook agents (CZ_STEP_COOK_AGENTS): the device cook acts for chosen agents inside the step.

The rule (include/cz_b200.h): every path gives, bit for bit, the composition heuristic_actions() -> overwrite the masked
columns -> step(), one step at a time.  Section 1 holds every path to that composition (a twin environment runs it), section
2 holds the device to the oracles (oracle/cz_policy.py decides for the masked agents on oracle/cz_oracle.py, the compiled
oracle steps beside it), section 3 holds episode statistics to a composition twin that keeps its own, sections 4 and 5
cover the one-launch closed loop, the full-size batch, CUDA graphs, changing roles and masked resets, section 6 the errors."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import cz_policy
from oracle.cz_oracle import OracleEnv, SpawnStream
from oracle.cz_oracle_c import COracleEnv
from tests.kitchens import kitchen, kitchen_config, plan_class, served_recipes, warp_group
from tests.test_gpu_random_kitchens import ARMS, N, _launches, _make

pytestmark = pytest.mark.gpu
RECIPES = ["TomatoLettuceSalad", "CarrotBanana"]


def _same(a, b, ctx):
    if a.dtype.is_floating_point:
        w = torch.int32 if a.element_size() == 4 else torch.int64
        a, b = a.contiguous().view(w), b.contiguous().view(w)
    assert a.shape == b.shape and torch.equal(a, b), ctx


def _bits(mask_b):
    """bool [N, A] -> int32 [N] bit mask"""
    A = mask_b.shape[1]
    return (mask_b.to(torch.int32) * torch.tensor([1 << i for i in range(A)], dtype=torch.int32, device=mask_b.device)).sum(1)


def _compose(twin, mask_b, acts, cook_recipes=None):
    """one step of the composition on `twin`: the merged actions it applied and the cook's raise bits under the mask"""
    cook, crashed = twin.heuristic_actions(cook_recipes)
    merged = torch.where(mask_b, cook, acts.to(torch.uint8))
    crash = crashed.to(torch.int32) & _bits(mask_b)
    twin.step(merged)
    return merged, crash


def _mask_b(spec, n, A):
    if isinstance(spec, torch.Tensor):
        return spec.cuda()
    m = torch.zeros((n, A), dtype=torch.bool, device="cuda")
    m[:, list(spec)] = True
    return m


# ---------------------------------------------------------------------------------------------------- 1. every path
PATH_KITCHENS = [32, 16, 68, 28, 20, 1017, 1002, 1003, 1142, 2, 13, 30]
COOK_ARMS = list(ARMS) + ["k8_keep", "dev_k8", "grid", "grid_k8_keep"]
MAX_STEPS, PHASE = 11, 8        # auto-reset every 11 steps; three masks of 8 steps each


def _cook_launches(arm, cls):
    """launches of one step (of 8 for the k8 arms) with cook agents: the warp kernel takes the cook in, every per-step path
    launches the merge kernel once per step (under device actions in place of the random-action kernel)"""
    packed = cls.startswith("packed")
    if arm in ("warp", "warp32"):
        return 1 if packed else 2
    if arm in ("k8", "k8_keep", "dev_k8"):
        return 1 if packed else 16
    if arm == "grid":                    # dynamics without rows (the warp kernel, or merge + generic kernel), then the grid
        return 2 if packed else 3
    if arm == "grid_k8_keep":            # eight single steps of grid mode
        return 16 if packed else 24
    if arm not in ARMS:
        return None
    base = _launches(arm, cls)
    return None if base is None else base + 1


@pytest.mark.parametrize("seed", PATH_KITCHENS)
def test_every_path_equals_the_composition(seed, monkeypatch, tmp_path):
    lp, mp, _ = kitchen(seed, str(tmp_path))
    cfg = kitchen_config(seed)
    A = cfg["A"]
    rng = np.random.default_rng(seed)
    rand_mask = torch.from_numpy(rng.random((N, A)) < 0.5)
    rand_mask[::5] = False                                   # environments without a cook
    specs = [[A - 1], list(range(A)), rand_mask]
    cook_recipes = list(reversed(cfg["recipes"])) if seed % 2 == 0 else None   # explicit cook recipes on half the kitchens
    for arm in COOK_ARMS:
        env_vars, kw = ARMS.get(arm, ({}, {}))
        kw = dict(kw)
        twin_kw = {}
        if arm.startswith("grid"):
            kw["obs_spaces"] = twin_kw["obs_spaces"] = ["grid"] * A
        common = dict(max_steps=MAX_STEPS, auto_reset=True)
        env = _make(lp, mp, cfg, seed, N, monkeypatch, env_vars, cook_agents=specs[0], cook_recipes=cook_recipes, **common, **kw)
        cls = plan_class(env.tables)
        if arm == "pipelined" and not cls.startswith("packed"):
            env.close()
            continue
        twin = _make(lp, mp, cfg, seed, N, monkeypatch, {}, **common, **twin_kw)
        env.reset(); twin.reset()
        acts = torch.from_numpy(rng.integers(0, env.tables.num_actions, size=(3 * PHASE, N, A)).astype(np.uint8)).cuda()
        K = 8 if "k8" in arm else 1
        keep = arm.endswith("keep")
        want_launches = _cook_launches(arm, cls)
        for ph in range(3):
            if ph:
                env.set_cook_agents(specs[ph])
            mb = _mask_b(specs[ph], N, A)
            for s0 in range(ph * PHASE, (ph + 1) * PHASE, K):
                ctx = f"kitchen {seed} ({cls}, A={A}) arm {arm} step {s0}"
                l0 = env.lib.cz_launch_count()
                if K > 1:
                    if arm == "dev_k8":
                        out = env.step_k(K, action_step=s0)
                    else:
                        out = env.step_k(K, actions=acts[s0:s0 + K], keep_all=keep)
                else:
                    out = env.step(acts[s0])
                    if arm == "pipelined":
                        env.wait()
                if want_launches is not None:
                    assert env.lib.cz_launch_count() - l0 == want_launches, ctx
                crash_or = torch.zeros(N, dtype=torch.int32, device="cuda")
                for j in range(K):
                    a = twin.random_actions(s0 + j).clone() if arm == "dev_k8" else acts[s0 + j]
                    merged, crash = _compose(twin, mb, a, cook_recipes)
                    crash_or |= crash
                    if keep:
                        o = twin.obs.float() if env.obs_dtype == torch.float32 else twin.obs
                        _same(out[0][j], o, ctx); _same(out[1][j], twin.reward, ctx)
                        _same(out[2][j], twin.terminated, ctx); _same(out[3][j], twin.truncated, ctx)
                        _same(env.actions_taken[j], merged, ctx)
                if not keep:
                    o = twin.obs.float() if env.obs_dtype == torch.float32 else twin.obs
                    _same(out[0], o, ctx); _same(out[1], twin.reward, ctx)
                    _same(out[2], twin.terminated, ctx); _same(out[3], twin.truncated, ctx)
                    _same(env.actions_taken, merged, ctx)
                _same(env.cook_step_crashed.to(torch.int32), crash_or, ctx)
                _same(env.error_flags, twin.error_flags, ctx)
                _same(env.state, twin.state, ctx)
        env.close(); twin.close()


_PROFILE = r"""
import json, os, sys
import torch
sys.path.insert(0, sys.argv[1])
from cooking_zoo_b200 import BatchedCookingEnv
out = {}
for name, n, env_vars, kw, k in [("warp", 2048, {}, {}, 1), ("k8", 2048, {}, {}, 8), ("lane", 2048, {"CZ_WARP_MAX_ENVS": "0"}, {}, 1),
                                 ("two", 32768, {}, {}, 1), ("f32", 8192, {}, {"obs_dtype": torch.float32}, 1),
                                 ("pipelined", 8192, {}, {"pipelined": True}, 1), ("lane_k4", 2048, {"CZ_WARP_MAX_ENVS": "0",
                                 "CZ_WARP_K_MAX_ENVS": "0"}, {}, 4)]:
    for cook in (False, True):
        os.environ.update(env_vars)
        env = BatchedCookingEnv(n, "coop_test", "example", 2, 25, ["TomatoLettuceSalad", "CarrotBanana"],
                                action_scheme="scheme3", auto_reset=True, cook_agents=[1] if cook else None, **kw)
        for v in env_vars:
            del os.environ[v]
        env.reset()
        a = env.random_actions(0)
        go = (lambda: env.step_k(k)) if k > 1 else (lambda: env.step(a))
        go(); env.wait(); torch.cuda.synchronize()
        l0 = env.lib.cz_launch_count()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            go(); env.wait()
            torch.cuda.synchronize()
        names = sorted({e.key[e.key.index("cz_"):].split("(")[0] for e in prof.key_averages() if "cz_" in e.key})
        out[name + ("_on" if cook else "_off")] = {"launches": env.lib.cz_launch_count() - l0, "kernels": names}
        env.close()
print(json.dumps(out))
"""


def test_launches_and_kernels_with_and_without_cook_agents():
    """off: the kernels of the default paths; on: the warp kernel's COOK instantiation in the same single launch, and one
    merge kernel (cz_policy_kernel<true>) per step on the per-step paths, which replaces the random-action kernel under
    CZ_STEP_DEVICE_ACTIONS.  torch.profiler runs in a process of its own."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", _PROFILE, root], cwd=root, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    print(out)
    for name in ("warp", "k8", "lane", "two", "f32", "pipelined", "lane_k4"):
        off, on = out[name + "_off"], out[name + "_on"]
        assert not any("policy" in k for k in off["kernels"]), (name, off)
        if name in ("warp", "k8"):
            assert off["launches"] == on["launches"] == 1, (name, off, on)
            assert off["kernels"] == ["cz_warp_kernel<2, 16, false, false>"], (name, off)
            assert on["kernels"] == ["cz_warp_kernel<2, 16, true, false>"], (name, on)
        elif name == "lane_k4":
            assert on["launches"] == off["launches"], (name, off, on)
            want = sorted((set(off["kernels"]) - {"cz_random_actions_kernel"}) | {"cz_policy_kernel<true>"})
            assert "cz_random_actions_kernel" in off["kernels"] and on["kernels"] == want, (name, off, on)
        else:
            assert on["launches"] == off["launches"] + 1, (name, off, on)
            assert on["kernels"] == sorted(off["kernels"] + ["cz_policy_kernel<true>"]), (name, off, on)


# ---------------------------------------------------------------------------------------------------- 2. oracles
ORACLE_KITCHENS = [(32, False), (16, False), (29, False), (28, True), (1, False), (49, False), (68, False), (117, False),
                   (77, False), (12, False), (189, False), (36, False)]
ORACLE_N, ORACLE_STEPS = 512, 60


def _oracle_lockstep(seed, generic, monkeypatch, tmp):
    lp, mp, level = kitchen(seed, str(tmp))
    cfg = dict(kitchen_config(seed))
    A = cfg["A"]
    served = served_recipes(level)
    assert served, seed
    cfg["recipes"] = [served[i % len(served)] for i in range(A)]
    rng = np.random.default_rng(seed)
    mask = rng.random((ORACLE_N, A)) < 0.6
    mask[::7] = False
    explicit = [served[(i + 1) % len(served)] for i in range(A)] if seed % 2 else None
    env = _make(lp, mp, cfg, seed, ORACLE_N, monkeypatch, {"CZ_GENERIC": "1"} if generic else {}, max_steps=200,
                recipe_pool=served, cook_agents=torch.from_numpy(mask), cook_recipes=explicit)
    t = env.tables
    names = t.recipe_names
    lids = rng.integers(0, t.num_layouts, size=ORACLE_N).astype(np.int32)
    rids = rng.integers(0, len(served), size=(ORACLE_N, A)).astype(np.uint8)
    rids = np.array([[names.index(served[r]) for r in row] for row in rids], np.uint8)
    env.reset(layout_ids=lids, recipe_ids=rids)

    def oracle(k, cls=OracleEnv):
        kw = dict(cfg["spawn"], spawn_stream=SpawnStream(seed, k, 1)) if cfg["spawn"] else {}
        return cls(t.layouts[lids[k]], [names[r] for r in rids[k]], 200, end_condition_all_dishes=cfg["end_all"],
                   action_scheme=cfg["scheme"], **kw)
    # the policy oracle reads the Python oracle's object graph; the compiled oracle steps beside it on the same actions
    oracles = {k: oracle(k) for k in range(ORACLE_N)}
    compiled = {k: oracle(k, COracleEnv) for k in range(ORACLE_N)}
    alive = set(oracles)
    counts = {}
    for s in range(ORACLE_STEPS):
        acts = rng.integers(0, t.num_actions, size=(ORACLE_N, A)).astype(np.uint8)
        merged, bits = acts.astype(np.int64), np.zeros(ORACLE_N, np.int64)
        for k in alive:
            want = cz_policy.heuristic_actions(oracles[k], explicit or [names[r] for r in rids[k]])
            for i in range(A):
                if mask[k, i]:
                    merged[k, i] = max(want[i], 0)
                    bits[k] |= (want[i] < 0) << i
                    counts[want[i]] = counts.get(want[i], 0) + 1
        obs, rew, term, _, _ = env.step(torch.from_numpy(acts))
        taken, crashed = env.actions_taken.cpu().numpy(), env.cook_step_crashed.cpu().numpy()
        obs, rew, term = obs.cpu().numpy(), rew.cpu().numpy(), term.cpu().numpy()
        for k in sorted(alive):
            ctx = f"kitchen {seed} env {k} step {s}"
            assert taken[k].tolist() == merged[k].tolist(), ctx
            assert int(crashed[k]) == int(bits[k]), ctx
            r, te, _, _ = oracles[k].step(merged[k].astype(np.uint8))
            assert np.array_equal(np.asarray(r, np.float64).view(np.uint64), rew[k].view(np.uint64)), ctx
            assert [int(v) for v in te] == list(term[k]), ctx
            cr, cte, _, _ = compiled[k].step(merged[k].astype(np.uint8))
            assert np.array_equal(cr.view(np.uint64), rew[k].view(np.uint64)) and list(cte) == list(term[k]), ctx
            rows = np.stack([compiled[k].observe(i) for i in range(A)])
            assert np.array_equal(rows.view(np.uint64), obs[k].view(np.uint64)), ctx
            if any(te):
                alive.discard(k)
    env.close()
    return counts


def test_cook_agents_against_the_oracles(monkeypatch, tmp_path):
    counts = {}
    for seed, generic in ORACLE_KITCHENS:
        for k, v in _oracle_lockstep(seed, generic, monkeypatch, tmp_path).items():
            counts[k] = counts.get(k, 0) + v
    print("masked cook decisions:", dict(sorted(counts.items())))
    assert {1, 2, 3, 4} <= set(counts) and counts.get(-1, 0) < sum(counts.values()) // 2


# ---------------------------------------------------------------------------------------------------- 3. statistics
STATS_KITCHENS = [(16, {}), (28, {}), (132, {}), (1002, {"CZ_WARP_GROUP": "32"}), (1003, {"CZ_WARP_GROUP": "32"}),
                  (68, {"CZ_WARP_MAX_ENVS": "0", "CZ_WARP_K_MAX_ENVS": "0"})]


@pytest.mark.parametrize("seed,env_vars", STATS_KITCHENS, ids=[str(s) for s, _ in STATS_KITCHENS])
def test_episode_statistics_equal_the_composition(seed, env_vars, monkeypatch, tmp_path):
    """cook agents with episode_stats=True against a composition twin that keeps its own statistics: single steps and
    step_k(8).  On the packed kitchens with more than 16 dynamic slots, or with CZ_WARP_GROUP=32, both run
    cz_warp_kernel<NA, 32, true, true>; the last kitchen runs the per-step paths (merge kernel, step, statistics kernel)."""
    lp, mp, _ = kitchen(seed, str(tmp_path))
    cfg = kitchen_config(seed)
    A = cfg["A"]
    rng = np.random.default_rng(seed)
    mask = torch.from_numpy(rng.random((N, A)) < 0.6)
    mask[::5] = False
    cook_recipes = list(reversed(cfg["recipes"])) if seed % 2 == 0 else None
    common = dict(max_steps=MAX_STEPS, auto_reset=True, episode_stats=True)
    env = _make(lp, mp, cfg, seed, N, monkeypatch, env_vars, cook_agents=mask, cook_recipes=cook_recipes, **common)
    twin = _make(lp, mp, cfg, seed, N, monkeypatch, {}, **common)
    if "CZ_WARP_MAX_ENVS" not in env_vars:
        assert plan_class(env.tables).startswith("packed") and (env_vars or warp_group(env.tables) == 32), seed
    env.reset(); twin.reset()
    env.clear_episode_stats(); twin.clear_episode_stats()
    mb = mask.cuda()
    acts = torch.from_numpy(rng.integers(0, env.tables.num_actions, size=(32, N, A)).astype(np.uint8)).cuda()
    for s0, K in [(0, 1), (1, 1), (2, 8), (10, 1), (11, 8), (19, 8), (27, 1), (28, 1), (29, 1)]:
        ctx = f"kitchen {seed} step {s0} K {K}"
        out = env.step(acts[s0]) if K == 1 else env.step_k(K, actions=acts[s0:s0 + K])
        for j in range(K):
            merged, _ = _compose(twin, mb, acts[s0 + j], cook_recipes)
        _same(env.actions_taken, merged, ctx)
        _same(out[1], twin.reward, ctx); _same(env.state, twin.state, ctx); _same(env.error_flags, twin.error_flags, ctx)
        a, b = env.episode_stats(), twin.episode_stats()
        for k in a:
            _same(a[k], b[k], f"{ctx} {k}")
        ta, tb = env.episode_totals(), twin.episode_totals()
        _same(ta[:4], tb[:4], ctx)
        torch.testing.assert_close(ta[4:], tb[4:], rtol=1e-12, atol=1e-9)       # summation order of the atomics
    assert int(env.episode_stats()["finished"].sum()) >= N, seed
    env.close(); twin.close()


# ---------------------------------------------------------------------------------------------------- 4. closed loop
def _coop(n, **kw):
    from cooking_zoo_b200 import BatchedCookingEnv
    return BatchedCookingEnv(n, "coop_test", "example", 2, kw.pop("max_steps", 20), RECIPES, action_scheme="scheme3",
                             auto_reset=True, seed=11, **kw)


@pytest.mark.parametrize("stats", [False, True])
def test_closed_loop_k_steps_in_one_launch(stats):
    n = 4096
    fused, single, twin = (_coop(n, cook_agents=[0, 1], episode_stats=stats), _coop(n, cook_agents=[0, 1], episode_stats=stats),
                           _coop(n))
    for e in (fused, single, twin):
        e.reset()
    l0 = fused.lib.cz_launch_count()
    out = fused.step_k(64, keep_all=True)
    assert fused.lib.cz_launch_count() - l0 == 1
    zeros = torch.zeros((n, 2), dtype=torch.uint8, device="cuda")
    mb = torch.ones((n, 2), dtype=torch.bool, device="cuda")
    crash_or = torch.zeros(n, dtype=torch.int32, device="cuda")
    for j in range(64):
        o, r, te, tu, _ = single.step(zeros)
        merged, crash = _compose(twin, mb, zeros)
        crash_or |= crash
        _same(single.actions_taken, merged, j); _same(single.cook_step_crashed.to(torch.int32), crash, j)
        _same(single.state, twin.state, j); _same(o, twin.obs, j); _same(r, twin.reward, j)
        _same(out[0][j], o, j); _same(out[1][j], r, j); _same(out[2][j], te, j); _same(out[3][j], tu, j)
        _same(fused.actions_taken[j], single.actions_taken, j)
    _same(fused.state, single.state, "state")
    _same(fused.cook_step_crashed.to(torch.int32), crash_or, "crashed")
    assert int(twin.state[twin.tables.num_dyn_slots + 2 + 5].min()) >= 3        # EPISODE row: episodes restarted in the launch
    if stats:
        a, b = fused.episode_stats(), single.episode_stats()
        for k in a:
            _same(a[k], b[k], k)
        assert int(a["finished"].sum()) >= 2 * n
    for e in (fused, single, twin):
        e.close()


# ---------------------------------------------------------------------------------------------------- 5. scale, graphs
def test_full_scale_in_place_and_pipelined_with_role_changes_and_masked_resets():
    n = 131072
    inplace, pipe, twin = _coop(n, cook_agents=[0], max_steps=15), _coop(n, cook_agents=[0], max_steps=15, pipelined=True), \
        _coop(n, max_steps=15)
    for e in (inplace, pipe, twin):
        e.reset()
    spec = [0]
    reset_mask = torch.from_numpy(np.arange(n) % 3 == 0)
    for s in range(20):
        if s == 8:                                              # roles change between calls
            spec = [1]
            inplace.set_cook_agents(spec); pipe.set_cook_agents(spec)
        if s == 13:                                             # a masked reset
            lids = twin.default_layout_ids(episode=5)
            for e in (inplace, pipe, twin):
                e.reset(layout_ids=lids, mask=reset_mask)
        a = twin.random_actions(s).clone()
        inplace.step(a)
        pipe.step(a); pipe.wait()
        merged, crash = _compose(twin, _mask_b(spec, n, 2), a)
        for name, e in (("in place", inplace), ("pipelined", pipe)):
            ctx = f"{name} step {s}"
            _same(e.obs, twin.obs, ctx); _same(e.reward, twin.reward, ctx)
            _same(e.terminated, twin.terminated, ctx); _same(e.truncated, twin.truncated, ctx)
            _same(e.state, twin.state, ctx); _same(e.error_flags, twin.error_flags, ctx)
            _same(e.actions_taken, merged, ctx); _same(e.cook_step_crashed.to(torch.int32), crash, ctx)
    for e in (inplace, pipe, twin):
        e.close()


@pytest.mark.parametrize("n", [2048, 20000])
def test_cuda_graph_equals_eager(n):
    def run(graph):
        env = _coop(n, cook_agents=[1], max_steps=6)
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
        out = {"state": env.state.clone(), "obs": env.obs.clone(), "taken": env.actions_taken.clone(),
               "crashed": env.cook_step_crashed.clone(), "reward": env.reward.clone()}
        env.close()
        return out
    eager, graph = run(False), run(True)
    for k in eager:
        _same(eager[k], graph[k], k)


# ---------------------------------------------------------------------------------------------------- 6. errors
def test_errors():
    import ctypes as C
    from cooking_zoo_b200 import _native, MixedAgentCookingEnv
    env, other = _coop(64), _coop(64)
    lib = env.lib
    env.reset()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    args = lambda flags, n=64, k=1: (env._handle, env.state.data_ptr(), env._actions.data_ptr(), env.obs.data_ptr(),
                                     env.reward.data_ptr(), env.terminated.data_ptr(), env.truncated.data_ptr(), None, n, k,
                                     flags, 0, 0, 0, s)
    COOK = _native.STEP_COOK_AGENTS
    assert lib.cz_step(*args(COOK)) == -1                                  # the flag with nothing attached
    assert b"cz_cook_attach" in lib.cz_last_error()
    mask = torch.full((64,), 1, dtype=torch.uint8, device="cuda")
    taken = torch.zeros((64, 2), dtype=torch.uint8, device="cuda")
    d = _native.CookDesc()
    d.n_envs, d.k_capacity, d.agent_mask, d.actions_taken = 64, 1, mask.data_ptr(), taken.data_ptr()
    assert lib.cz_cook_attach(env._handle, other._policy_handle(), C.byref(d)) == -1    # a policy of other tables
    assert lib.cz_cook_attach(env._handle, None, C.byref(d)) == -1
    policy = env._policy_handle()
    for field, bad in (("agent_mask", None), ("actions_taken", None), ("n_envs", 0), ("k_capacity", 0)):
        d2 = _native.CookDesc()
        d2.n_envs, d2.k_capacity, d2.agent_mask, d2.actions_taken = 64, 1, mask.data_ptr(), taken.data_ptr()
        setattr(d2, field, bad)
        assert lib.cz_cook_attach(env._handle, policy, C.byref(d2)) == -1, field
    assert lib.cz_cook_attach(env._handle, policy, C.byref(d)) == 0
    assert lib.cz_step(*args(COOK, 32)) == -1                              # n_envs differs from the attached one
    assert b"n_envs" in lib.cz_last_error()
    assert lib.cz_step(*args(COOK, 0)) == -1 and lib.cz_step(*args(0, 0)) == 0   # an empty batch differs too
    assert lib.cz_step(*args(COOK | _native.STEP_KEEP_ALL, 64, 2)) == -1   # KEEP_ALL beyond k_capacity
    assert b"k_capacity" in lib.cz_last_error()
    host = [np.zeros(64 * 2 * env.obs_len), np.zeros(64 * 2), np.zeros(128, np.uint8), np.zeros(128, np.uint8)]
    acts = np.zeros(128, np.uint8)
    assert lib.cz_step_host(env._handle, env.state.data_ptr(), acts.ctypes.data, host[0].ctypes.data, host[1].ctypes.data,
                            host[2].ctypes.data, host[3].ctypes.data, 64, COOK, 0, 0, s) == -1
    assert lib.cz_step(*args(COOK)) == 0
    torch.cuda.synchronize()
    assert lib.cz_cook_attach(env._handle, None, None) == 0                # detach
    assert lib.cz_step(*args(COOK)) == -1
    with pytest.raises(_native.NativeError):
        env.set_cook_agents([0])
    with pytest.raises(ValueError):
        _coop(64, cook_agents=[2])
    with pytest.raises(ValueError):
        _coop(64, cook_agents=[-1])
    with pytest.raises(ValueError):
        _coop(64, cook_agents=torch.ones((63, 2), dtype=torch.bool))
    with pytest.raises(ValueError):
        _coop(64, cook_agents=[0], cook_recipes=["TomatoLettuceSalad", "NoSuchRecipe"])
    cooked = _coop(64, cook_agents=[0])
    with pytest.raises(ValueError):
        cooked.set_cook_agents([5])
    with pytest.raises(NotImplementedError):
        MixedAgentCookingEnv([1, 2, 2], "coop_test", "example", 20, RECIPES, action_scheme="scheme3", cook_agents=[0])
    for e in (env, other, cooked):
        e.close()
