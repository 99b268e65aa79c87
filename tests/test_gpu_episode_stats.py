"""GPU: episode statistics (BatchedCookingEnv(episode_stats=True), CZ_STEP_EPISODE_STATS) against oracle/cz_stats.py.

The per-environment record is compared bit for bit, after every call, with episode_stats_from_trace over the rewards and
post-step rows of a statistics-off twin that steps one step at a time with the same seed; the twin's outputs and state
must equal the statistics-on environment's bit for bit on every path the library can take."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import cz_stats
from tests.kitchens import DEVICE_KITCHENS, kitchen, kitchen_config, plan_class
from tests.replay import golden_files, load_golden, package_recipes
from tests.test_gpu_random_kitchens import ARMS, _make

pytestmark = pytest.mark.gpu
N = 3001
STEPS = 40
MAX_STEPS = 12
STAT_ARMS = dict(ARMS, k8_keep=({}, {}), grid=({}, {}))
DEV_KEYS = (("return", "ret"), ("last_return", "last_ret"), ("last_length", "last_len"), ("last_served", "last_served"),
            ("last_success", "last_success"), ("finished", "finished"))


def _rows(env):
    """post-step (EPISODE, t, done, roots [N, R]) of the current state, on the host"""
    from cooking_zoo_b200.tables import ROW_EPISODE, ROW_MARKS, ROW_TINFO
    t = env.tables
    base = t.num_dyn_slots + t.num_agents
    st = env.state.cpu().numpy().view(np.uint32)
    tt, done, roots = cz_stats.decode_misc(st[base + ROW_TINFO], st[base + ROW_MARKS], t.num_recipes)
    return st[base + ROW_EPISODE], tt, done, roots


def _feed(rec, twin, end_all, reward=None):
    """one step of the oracle rule from the twin's post-step rows and rewards"""
    ep, t, done, roots = _rows(twin)
    r = (twin.reward if reward is None else reward).cpu().numpy()
    return cz_stats.episode_stats_from_trace(r[None], ep[None], t[None], done[None], roots[None], end_all, record=rec)


def _start(env):
    """the oracle record of a freshly constructed environment (cleared on the all-zero state)"""
    n, A = env.num_envs, env.num_agents
    return cz_stats.clear(cz_stats.new_record(n, A), np.zeros(n), np.zeros(n))


def _assert_record(env, rec, ctx, internal=True):
    st = env.episode_stats()
    for dk, ok in DEV_KEYS:
        got, want = st[dk].cpu().numpy(), rec[ok]
        if got.dtype == np.float64:
            got, want = got.view(np.uint64), want.view(np.uint64)
        bad = (got != want.astype(got.dtype))
        if bad.ndim > 1:
            bad = bad.any(-1)
        if bad.any():
            e = int(np.flatnonzero(bad)[0])
            raise AssertionError(f"{ctx}: {dk} differs at environments {np.flatnonzero(bad)[:8].tolist()}: env {e} got "
                                 f"{st[dk][e].tolist()} want {rec[ok][e].tolist()}")
    if internal:
        assert np.array_equal(env._stats["episode"].cpu().numpy().view(np.uint32), rec["episode"]), ctx
        assert np.array_equal(env._stats["open"].cpu().numpy(), rec["open"]), ctx
    tot = env.episode_totals().cpu().numpy()
    assert np.array_equal(tot[:4], rec["totals"][:4]), (ctx, tot, rec["totals"])
    np.testing.assert_allclose(tot[4:], rec["totals"][4:], rtol=1e-12, atol=1e-9, err_msg=ctx)


def _same(a, b, ctx):
    assert a.dtype == b.dtype and a.shape == b.shape, ctx
    w = {8: torch.int64, 4: torch.int32, 1: torch.uint8}[a.element_size()]
    assert torch.equal(a.contiguous().view(w), b.contiguous().view(w)), ctx


# ---------------------------------------------------------------------------------------------------- 1. golden replay
@pytest.mark.parametrize("kernel", ["warp", "lane"])
@pytest.mark.parametrize("path", golden_files(), ids=lambda p: p.split("/")[-1][:-4])
def test_stats_replay_golden(path, kernel, monkeypatch):
    """"return" is the running float64 sum of the reference's recorded rewards after every step; a trace that finishes
    latches its length, returns and served recipes"""
    from cooking_zoo_b200 import BatchedCookingEnv
    if kernel == "lane":
        monkeypatch.setenv("CZ_WARP_MAX_ENVS", "0")
    g = load_golden(path)
    cfg = g["config"]
    n, A = len(g["layouts"]), cfg["num_agents"]
    if (np.asarray(g.get("raised", -np.ones(n))) >= 0).any():
        pytest.skip("trace ends where the reference raised")
    kw = {}
    sp = cfg.get("spawn")
    if sp:
        kw = dict(agent_respawn_rate=sp["respawn"], agent_despawn_rate=sp["despawn"], grace_period=sp["grace"], seed=sp["seed"])
    with package_recipes(cfg):
        env = BatchedCookingEnv(n, cfg["level"], cfg["meta_file"], A, cfg["max_steps"], cfg["recipes"],
                                end_condition_all_dishes=cfg["end_all"], reward_scheme=cfg["reward_scheme"],
                                action_scheme=cfg.get("action_scheme", "scheme3"), layouts=g["layouts"],
                                episode_stats=True, **kw)
    env.reset(layout_ids=np.arange(n))
    run = np.zeros((n, A))
    for t in range(g["actions"].shape[1]):
        live = [k for k in range(n) if t < g["length"][k]]
        if not live:
            break
        for k in live:
            for i in range(A):
                if g["teleport"][k, t, i, 0] >= 0:
                    env.teleport(k, i, *map(int, g["teleport"][k, t, i]))
        env.step(torch.from_numpy(g["actions"][:, t].astype(np.uint8)))
        got = env.episode_stats()["return"].cpu().numpy()
        for k in live:
            run[k] = run[k] + g["reward"][k, t]
            assert np.array_equal(got[k].view(np.uint64), run[k].view(np.uint64)), f"{path} trace {k} step {t}"
    st = {k: v.cpu().numpy() for k, v in env.episode_stats().items()}
    for k in range(n):
        L = int(g["length"][k])
        fin = L == cfg["max_steps"] or bool(g["term"][k, L - 1].any())
        assert st["finished"][k] == int(fin), (path, k)
        if fin:
            roots = (np.asarray(g["marks"][k, L]) & 1).astype(bool)
            served = int(roots.sum())
            assert st["last_length"][k] == L, (path, k)
            assert np.array_equal(st["last_return"][k].view(np.uint64), run[k].view(np.uint64)), (path, k)
            assert st["last_served"][k] == served, (path, k)
            assert st["last_success"][k] == int(served == len(roots) if cfg["end_all"] else served > 0), (path, k)
    env.close()


# ---------------------------------------------------------------------------------------------------- 2. every path
def _pair(lp, mp, cfg, seed, arm, monkeypatch, n=N):
    env_vars, kw = STAT_ARMS[arm]
    kw = dict(kw)
    if arm == "grid":
        kw["obs_spaces"] = ["grid"] * cfg["A"]
    common = dict(max_steps=MAX_STEPS, auto_reset=True)
    on = _make(lp, mp, cfg, seed, n, monkeypatch, env_vars, episode_stats=True, **common, **kw)
    twin = _make(lp, mp, cfg, seed, n, monkeypatch, {}, **common)
    return on, twin


def _obs_like(on, twin_obs):
    return twin_obs.float() if on.obs_dtype == torch.float32 else twin_obs


@pytest.mark.parametrize("seed", DEVICE_KITCHENS)
def test_every_path_keeps_the_oracle_statistics(seed, monkeypatch, tmp_path):
    lp, mp, _ = kitchen(seed, str(tmp_path))
    cfg = kitchen_config(seed)
    A = cfg["A"]
    for arm in STAT_ARMS:
        on, twin = _pair(lp, mp, cfg, seed, arm, monkeypatch)
        if arm == "pipelined" and not plan_class(on.tables).startswith("packed"):
            on.close(); twin.close()
            continue
        ctx0 = f"kitchen {seed} arm {arm}"
        on.reset(); twin.reset()
        rec = _start(on)
        rng = np.random.default_rng(seed)
        acts = torch.from_numpy(rng.integers(0, on.tables.num_actions, size=(STEPS, N, A)).astype(np.uint8)).cuda()
        K = 8 if arm.startswith("k8") else 1
        for s0 in range(0, STEPS, K):
            ctx = f"{ctx0} step {s0}"
            if K > 1:
                out = on.step_k(K, actions=acts[s0:s0 + K], keep_all=arm == "k8_keep")
            else:
                out = on.step(acts[s0])
                if arm == "pipelined":
                    on.wait()
            for j in range(K):
                o, r, te, tu, _ = twin.step(acts[s0 + j])
                rec = _feed(rec, twin, cfg["end_all"])
                if arm == "k8_keep":
                    _same(out[0][j], o, ctx); _same(out[1][j], r, ctx); _same(out[2][j], te, ctx); _same(out[3][j], tu, ctx)
            if arm != "k8_keep":
                if arm != "grid":
                    _same(out[0], _obs_like(on, twin.obs), ctx)
                _same(out[1], twin.reward, ctx); _same(out[2], twin.terminated, ctx); _same(out[3], twin.truncated, ctx)
            _same(on.error_flags, twin.error_flags, ctx)
            _same(on.state, twin.state, ctx)
            _assert_record(on, rec, ctx)
        assert rec["finished"].sum() >= N, ctx0           # many episodes finished
        on.close(); twin.close()


def test_full_scale_with_device_actions():
    """131072 two-agent coop_test environments, device random actions, max_steps 25, auto-reset: the default dispatch"""
    from cooking_zoo_b200 import BatchedCookingEnv
    n = 131072
    mk = lambda **kw: BatchedCookingEnv(n, "coop_test", "example", 2, 25, ["TomatoLettuceSalad", "CarrotBanana"],
                                        action_scheme="scheme3", auto_reset=True, seed=7, **kw)
    on, twin = mk(episode_stats=True), mk()
    on.reset(); twin.reset()
    rec = _start(on)
    for s in range(60):
        a = twin.random_actions(s)
        o, r, te, tu, _ = on.step(a)
        twin.step(a)
        rec = _feed(rec, twin, False)
        _same(o, twin.obs, s); _same(r, twin.reward, s); _same(on.state, twin.state, s)
        if s % 10 == 9 or s == 24:
            _assert_record(on, rec, f"step {s}")
    assert rec["finished"].sum() >= 2 * n
    on.close(); twin.close()


# ---------------------------------------------------------------------------------------------------- 3. launches
_PROFILE = r"""
import json, sys
import torch
sys.path.insert(0, sys.argv[1])
from cooking_zoo_b200 import BatchedCookingEnv
out = {}
for name, n, env_vars, kw, k in [("warp", 2048, {}, {}, 1), ("k8", 2048, {}, {}, 8), ("lane", 2048, {"CZ_WARP_MAX_ENVS": "0"}, {}, 1),
                                 ("two", 32768, {}, {}, 1), ("f32", 8192, {}, {"obs_dtype": torch.float32}, 1),
                                 ("pipelined", 8192, {}, {"pipelined": True}, 1), ("lane_k4", 2048, {"CZ_WARP_MAX_ENVS": "0",
                                 "CZ_WARP_K_MAX_ENVS": "0"}, {}, 4)]:
    import os
    for stats in (False, True):
        os.environ.update(env_vars)
        env = BatchedCookingEnv(n, "coop_test", "example", 2, 25, ["TomatoLettuceSalad", "CarrotBanana"],
                                action_scheme="scheme3", auto_reset=True, episode_stats=stats, **kw)
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
        out[name + ("_on" if stats else "_off")] = {"launches": env.lib.cz_launch_count() - l0, "kernels": names}
        env.close()
print(json.dumps(out))
"""


def test_launches_with_and_without_statistics():
    """statistics off: the kernels of the default path (the warp kernel's STATS = false instantiation); on: one more
    kernel per step, cz_stats_kernel, on the per-step paths and none on the warp kernel.  torch.profiler runs in a process
    of its own, so that this test leaves the profiler state of the test process as it was."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", _PROFILE, root], cwd=root, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    print(out)
    steps = {"k8": 1, "lane_k4": 4}
    for name in ("warp", "k8", "lane", "two", "f32", "pipelined", "lane_k4"):
        off, on = out[name + "_off"], out[name + "_on"]
        assert not any("stats" in k for k in off["kernels"]), (name, off)
        if name in ("warp", "k8"):
            assert off["launches"] == on["launches"] == 1, (name, off, on)
            assert len(off["kernels"]) == 1 and off["kernels"][0].startswith("cz_warp_kernel<2, "), (name, off)
            assert on["kernels"] == [off["kernels"][0].replace(", false>", ", true>")] != off["kernels"], (name, on)
        else:
            assert on["launches"] == off["launches"] + steps.get(name, 1), (name, off, on)
            assert on["kernels"] == sorted(off["kernels"] + ["cz_stats_kernel<2>"]), (name, off, on)


# ---------------------------------------------------------------------------------------------------- 4. semantics
def _coop(n, **kw):
    from cooking_zoo_b200 import BatchedCookingEnv
    kw.setdefault("max_steps", 10)
    return BatchedCookingEnv(n, "coop_test", "example", 2, kw.pop("max_steps"), ["TomatoLettuceSalad", "CarrotBanana"],
                             action_scheme="scheme3", seed=3, **kw)


@pytest.mark.parametrize("n", [1000, 40000])
def test_masked_reset_clear_and_stepping_past_the_end(n):
    """no auto-reset: stepping past the end latches once; a masked reset mid-run drops the partial episodes it hits;
    clear_episode_stats() mid-episode counts only episodes that start afterwards"""
    on, twin = _coop(n, episode_stats=True), _coop(n)
    on.reset(); twin.reset()
    rec = _start(on)
    mask = (np.arange(n) % 3 == 0)
    for s in range(30):
        if s == 4:                                           # masked reset mid-episode
            lids = on.default_layout_ids(episode=1)
            on.reset(layout_ids=lids, mask=mask); twin.reset(layout_ids=lids, mask=mask)
        if s == 7:                                           # a new counting window in the middle of episodes
            on.clear_episode_stats()
            ep, t, _, _ = _rows(twin)
            rec = cz_stats.clear(rec, ep, t)
        if s == 15:                                          # everybody starts over; the cleared window counts these whole
            on.reset(); twin.reset()
        a = twin.random_actions(s)
        on.step(a); twin.step(a)
        rec = _feed(rec, twin, False)
        _same(on.state, twin.state, s)
        _assert_record(on, rec, f"n {n} step {s}")
    assert rec["finished"].sum() == n and (rec["finished"] == 1).all()   # the second episodes finished at max_steps, once
    tot = on.episode_totals(clear=True)
    assert tot[0].item() == n and on.episode_totals()[0].item() == 0.0
    on.close(); twin.close()


def test_cuda_graph_equals_eager():
    def run(graph):
        env = _coop(20000, auto_reset=True, episode_stats=True, max_steps=6)
        env.reset()
        a = env.random_actions(0)
        if graph:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                env.step(a)                                  # warm-up outside the capture
            torch.cuda.current_stream().wait_stream(s)
            env.reset()
            env.clear_episode_stats()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for _ in range(20):
                    env.step(a)
            g.replay()
        else:
            env.step(a)
            env.reset()
            env.clear_episode_stats()
            for _ in range(20):
                env.step(a)
        torch.cuda.synchronize()
        out = {k: v.clone() for k, v in env.episode_stats().items()}
        out["totals"] = env.episode_totals()
        out["state"] = env.state.clone()
        env.close()
        return out
    eager, graph = run(False), run(True)
    assert eager["finished"].sum().item() > 20000
    for k in eager:
        if k == "totals":
            assert torch.equal(eager[k][:4], graph[k][:4])
            torch.testing.assert_close(eager[k][4:], graph[k][4:], rtol=1e-12, atol=1e-9)
        else:
            _same(eager[k], graph[k], k)


def test_mixed_population_against_its_groups():
    from cooking_zoo_b200.mixed import MixedAgentCookingEnv
    counts = np.array([1, 2, 2, 1, 2] * 200)
    mix = MixedAgentCookingEnv(counts, "coop_test", "example", 8, ["TomatoLettuceSalad", "CarrotBanana"],
                               action_scheme="scheme3", auto_reset=True, episode_stats=True)
    mix.reset()
    for s in range(20):
        mix.step(torch.randint(0, 5, (len(counts), 2), generator=torch.Generator().manual_seed(s), dtype=torch.uint8))
    st = mix.episode_stats()
    tot = torch.zeros(6, dtype=torch.float64, device="cuda")
    for a, g in mix.groups.items():
        idx = mix.index[a]
        gs = g.episode_stats()
        for k, v in gs.items():
            if v.dim() == 2:
                _same(st[k][idx, :a], v, k)
                assert (st[k][idx, a:] == 0).all(), k
            else:
                _same(st[k][idx], v, k)
        tot[:4 + a] += g.episode_totals()
    assert st["finished"].sum().item() > len(counts)
    assert torch.equal(mix.episode_totals(), tot)
    assert mix.episode_totals_names == ["episodes", "length", "served", "success", "return:player_0", "return:player_1"]
    mix.close()


def test_despawn_and_respawn():
    """agents that despawn and respawn: relevant agents change, the record follows the twin's rewards"""
    for env_vars in ({}, {"CZ_WARP_MAX_ENVS": "0"}):
        os.environ.update(env_vars)
        try:
            kw = dict(agent_respawn_rate=0.3, agent_despawn_rate=0.2, grace_period=2, auto_reset=True, max_steps=15)
            on, twin = _coop(3000, episode_stats=True, **kw), _coop(3000, **kw)
        finally:
            for v in env_vars:
                del os.environ[v]
        on.reset(); twin.reset()
        rec = _start(on)
        for s in range(40):
            a = twin.random_actions(s)
            on.step(a); twin.step(a)
            rec = _feed(rec, twin, False)
            _same(on.state, twin.state, s); _same(on.reward, twin.reward, s)
        _assert_record(on, rec, f"spawn {env_vars}")
        on.close(); twin.close()


def test_abi_errors():
    import ctypes as C
    from cooking_zoo_b200 import _native
    env = _coop(64)
    lib = env.lib
    with pytest.raises(_native.NativeError):
        env.episode_stats()
    with pytest.raises(_native.NativeError):
        env.episode_totals()
    with pytest.raises(_native.NativeError):
        env.clear_episode_stats()
    env.reset()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    args = lambda flags, n=64: (env._handle, env.state.data_ptr(), env._actions.data_ptr(), env.obs.data_ptr(),
                                env.reward.data_ptr(), env.terminated.data_ptr(), env.truncated.data_ptr(), None, n, 1, flags,
                                0, 0, 0, s)
    assert lib.cz_step(*args(_native.STEP_EPISODE_STATS)) == -1                 # the flag without attached buffers
    assert b"cz_stats_attach" in lib.cz_last_error()
    assert lib.cz_stats_clear(env._handle, env.state.data_ptr(), 64, s) == -1
    env._attach_episode_stats()
    assert lib.cz_step(*args(_native.STEP_EPISODE_STATS, 32)) == -1             # n_envs differs from the attached one
    assert b"n_envs" in lib.cz_last_error()
    assert lib.cz_stats_clear(env._handle, env.state.data_ptr(), 32, s) == -1
    d = _native.StatsDesc()
    d.n_envs = 64
    assert lib.cz_stats_attach(env._handle, C.byref(d)) == -1                   # null fields
    d2 = _native.StatsDesc()
    for f, _ in _native.StatsDesc._fields_[1:]:
        setattr(d2, f, env._stats["return"].data_ptr())
    d2.n_envs = 0
    assert lib.cz_stats_attach(env._handle, C.byref(d2)) == -1                  # n_envs < 1
    assert lib.cz_step(*args(_native.STEP_EPISODE_STATS)) == 0                  # a failed attach keeps the old buffers
    assert lib.cz_stats_attach(env._handle, None) == 0                          # detach
    assert lib.cz_step(*args(_native.STEP_EPISODE_STATS)) == -1
    assert lib.cz_step(*args(0)) == 0
    torch.cuda.synchronize()
    env.close()
