"""GPU: the grid observation (cz_observe_grid, obs_spaces=["grid"] * A) against oracle/cz_grid.py.

The device grid is compared with grid_from_state of the reference-recorded golden states, of the compiled oracle's states
(CBatch) on random kitchens and at full scale, and of the device's own exported state; a grid-mode environment and a
feature-vector twin with the same seed must step identically."""
import numpy as np
import pytest
import torch

from oracle.cz_grid import grid_from_states
from tests.kitchens import DEVICE_KITCHENS, kitchen, kitchen_config
from tests.replay import golden_files, load_golden, package_recipes

pytestmark = pytest.mark.gpu
RECIPES = ["TomatoLettuceSalad", "CarrotBanana"]


def _coop(n, A=2, **kw):
    from cooking_zoo_b200 import BatchedCookingEnv
    kw.setdefault("obs_spaces", ["grid"] * A)
    return BatchedCookingEnv(n, "coop_test", "example", A, kw.pop("max_steps", 400), RECIPES[:A],
                             end_condition_all_dishes=True, action_scheme="scheme3", **kw)


def _meta(env):
    return env.tables.layouts[0]["meta"]


def _own_grid(env):
    """grid_from_state of the device's own exported state: uint8 [N, A, C, H, W]"""
    t = env.tables
    return torch.from_numpy(grid_from_states(env.export_state(), _meta(env), t.num_agents, t.width, t.height))


def _assert_grid(got, want, ctx):
    got, want = got.cpu(), torch.as_tensor(want).cpu()
    assert got.shape == want.shape, (ctx, got.shape, want.shape)
    bad = (got != want).reshape(got.shape[0], -1).any(1)
    if bool(bad.any()):
        e = int(bad.nonzero()[0])
        idx = (got[e] != want[e]).nonzero()[0].tolist()
        raise AssertionError(f"{ctx}: environments {bad.nonzero().flatten()[:8].tolist()} differ; env {e} first at "
                             f"[observer, channel, y, x] = {idx}: got {int(got[e][tuple(idx)])} want {int(want[e][tuple(idx)])}")


# ---------------------------------------------------------------------------------------------------- 1. golden replay
@pytest.mark.parametrize("kernel", ["warp", "lane"])
@pytest.mark.parametrize("path", golden_files(), ids=lambda p: p.split("/")[-1][:-4])
def test_grid_replays_golden(path, kernel, monkeypatch):
    """at reset and after every step (teleports included) the device grid equals grid_from_state of the state recorded from
    the reference; "lane" forces the lane-per-environment kernels for the dynamics"""
    from cooking_zoo_b200 import BatchedCookingEnv
    if kernel == "lane":
        monkeypatch.setenv("CZ_WARP_MAX_ENVS", "0")
    g = load_golden(path)
    cfg = g["config"]
    n, A = len(g["layouts"]), cfg["num_agents"]
    kw = {}
    sp = cfg.get("spawn")
    if sp:
        kw = dict(agent_respawn_rate=sp["respawn"], agent_despawn_rate=sp["despawn"], grace_period=sp["grace"], seed=sp["seed"])
    with package_recipes(cfg):
        env = BatchedCookingEnv(n, cfg["level"], cfg["meta_file"], A, cfg["max_steps"], cfg["recipes"],
                                end_condition_all_dishes=cfg["end_all"], reward_scheme=cfg["reward_scheme"],
                                action_scheme=cfg.get("action_scheme", "scheme3"), layouts=g["layouts"],
                                obs_spaces=["grid"] * A, **kw)

    wants = []
    for k, lay in enumerate(g["layouts"]):       # every recorded state of trace k
        states = [{key: g[key][k, t] for key in ("agents", "objs", "statics")} for t in range(int(g["length"][k]) + 1)]
        wants.append(grid_from_states(states, lay["meta"], A, lay["width"], lay["height"]))
    grid = env.reset(layout_ids=np.arange(n)).cpu().numpy()
    for k in range(n):
        assert np.array_equal(grid[k], wants[k][0]), f"{path} trace {k} reset"
    for t in range(g["actions"].shape[1]):
        live = [k for k in range(n) if t < g["length"][k]]
        if not live:
            break
        for k in live:
            for i in range(A):
                if g["teleport"][k, t, i, 0] >= 0:
                    env.teleport(k, i, *map(int, g["teleport"][k, t, i]))
        grid = env.step(torch.from_numpy(g["actions"][:, t].astype(np.uint8)))[0].cpu().numpy()
        for k in live:
            assert np.array_equal(grid[k], wants[k][t + 1]), f"{path} trace {k} step {t}"


# ---------------------------------------------------------------------------------------------------- 2. random kitchens
def _kitchen_env(lp, mp, cfg, seed, n, **kw):
    from cooking_zoo_b200 import BatchedCookingEnv
    return BatchedCookingEnv(n, lp, mp, cfg["A"], 40, cfg["recipes"], end_condition_all_dishes=cfg["end_all"],
                             action_scheme=cfg["scheme"], layout_pool_size=16, layout_seed=seed, seed=seed,
                             **(cfg["spawn"] or {}), **kw)


def test_random_kitchens_include_odd_grid_sizes(tmp_path):
    from cooking_zoo_b200.grid import grid_channels
    from cooking_zoo_b200.tables import compile_tables
    odd = []
    for seed in DEVICE_KITCHENS:
        lp, mp, _ = kitchen(seed, str(tmp_path))
        cfg = kitchen_config(seed)
        t = compile_tables(lp, mp, cfg["A"], 40, cfg["recipes"], layout_pool_size=2)
        if cfg["A"] * len(grid_channels(t)) * t.width * t.height % 2:
            odd.append(seed)
    assert len(odd) >= 2, odd


@pytest.mark.parametrize("seed", DEVICE_KITCHENS)
def test_grid_on_random_kitchens(seed, tmp_path):
    """3001 environments, 40 steps: the grid-mode environment and its feature-vector twin step identically (state, rewards,
    flags, error_flags) and the grid equals grid_from_state of CBatch's state (every environment at steps 0, 1, 20 and 40,
    64 sampled ones at the other steps)"""
    from oracle.cz_oracle_c import CBatch
    n, steps = 3001, 40
    lp, mp, _ = kitchen(seed, str(tmp_path))
    cfg = kitchen_config(seed)
    A = cfg["A"]
    env = _kitchen_env(lp, mp, cfg, seed, n, obs_spaces=["grid"] * A)
    twin = _kitchen_env(lp, mp, cfg, seed, n)
    t = env.tables
    lids = env.default_layout_ids().cpu().numpy()
    cpu = CBatch([t.layouts[l] for l in lids], [cfg["recipes"]] * n, 40, end_condition_all_dishes=cfg["end_all"],
                 action_scheme=cfg["scheme"], **(cfg["spawn"] or {}))
    if cfg["spawn"]:
        for k, e in enumerate(cpu.envs):
            cpu.lib.czo_set_stream(e.h, seed, k, 1)
    meta = t.layouts[0]["meta"]
    sample = np.random.default_rng(seed).choice(n, 64, replace=False)

    def check(grid, s, live):
        envs = np.arange(n) if s in (0, 1, 20, 40) else sample
        envs = envs[live[envs]]
        want = grid_from_states([cpu.envs[k].export_state() for k in envs], meta, A, t.width, t.height)
        _assert_grid(grid[torch.from_numpy(envs).cuda()], want, f"kitchen {seed} (A={A}) step {s}")

    grid = env.reset(layout_ids=lids)
    twin.reset(layout_ids=lids)
    live = np.ones(n, bool)
    check(grid, 0, live)
    rng = np.random.default_rng(seed)
    for s in range(1, steps + 1):
        act = rng.integers(0, t.num_actions, size=(n, A)).astype(np.uint8)
        grid, r, te, tu, _ = env.step(torch.from_numpy(act))
        _, r2, te2, tu2, _ = twin.step(torch.from_numpy(act))
        ctx = f"kitchen {seed} step {s}"
        assert torch.equal(env.state, twin.state), ctx
        assert torch.equal(r.view(torch.int64), r2.view(torch.int64)), ctx
        assert torch.equal(te, te2) and torch.equal(tu, tu2), ctx
        assert torch.equal(env.error_flags, twin.error_flags), ctx
        _, _, cte, ctu = cpu.step(act)
        check(grid, s, live)
        live &= ~cte.astype(bool).any(1)       # the episode is over: no auto-reset here, compare the running ones
    assert live.sum() > 0


# ---------------------------------------------------------------------------------------------------- 3. scale
def test_grid_at_scale_with_auto_reset():
    """131072 two-agent coop_test environments, 30 auto-reset steps of random actions: at the last step every grid equals
    grid_from_state of CBatch's state (environments whose episode ended are compared with the device's own state)"""
    from oracle.cz_oracle_c import CBatch
    n, steps = 131072, 30
    env = _coop(n, auto_reset=True, seed=3)
    lids = env.default_layout_ids().cpu().numpy()
    env.reset(layout_ids=lids)
    cpu = CBatch([env.tables.layouts[l] for l in lids], [RECIPES] * n, 400, end_condition_all_dishes=True)
    ended = np.zeros(n, bool)
    for s in range(steps):
        act = env.random_actions(s)
        grid = env.step(act)[0]
        _, _, cte, ctu = cpu.step(act.cpu().numpy())
        ended |= (cte | ctu).astype(bool).any(1)
    got = grid.cpu()
    keep = np.flatnonzero(~ended)
    assert len(keep) > n // 2
    want = grid_from_states([cpu.envs[k].export_state() for k in keep], _meta(env), 2, 7, 7)
    _assert_grid(got[torch.from_numpy(keep)], want, "131072 envs, step 30, running episodes")
    _assert_grid(got, _own_grid(env), "131072 envs, step 30, device state")


# ---------------------------------------------------------------------------------------------------- 4. sizes, alignment
@pytest.mark.parametrize("A", [1, 2])
@pytest.mark.parametrize("n", [1, 31, 33, 129, 20483])
def test_grid_ragged_batches(n, A):
    """one-agent coop_test grids are 1911 bytes (odd), two-agent ones 4508: every block boundary falls off 16 bytes"""
    env = _coop(n, A, seed=n)
    grid = env.reset(layout_ids=env.default_layout_ids())
    _assert_grid(grid, _own_grid(env), f"n={n} A={A} reset")
    for s in range(3):
        grid = env.step(env.random_actions(s))[0]
        _assert_grid(grid, _own_grid(env), f"n={n} A={A} step {s}")


@pytest.mark.parametrize("A,n", [(1, 33), (2, 31), (2, 3001)])
def test_grid_k_steps_equal_single_steps(A, n):
    """step_k(8, keep_all=True) == 8 single steps (A=1, n=33: a step's block of 33 x 1911 bytes is odd); step_k(8) keeps
    the last of them"""
    a, b, c = (_coop(n, A, seed=11) for _ in range(3))
    lids = a.default_layout_ids()
    for e in (a, b, c):
        e.reset(layout_ids=lids)
    acts = torch.randint(0, 5, (8, n, A), dtype=torch.uint8, device="cuda")
    gk, rk, tk, uk, _ = a.step_k(8, actions=acts, keep_all=True)
    assert gk.shape == (8,) + tuple(a.obs.shape)
    for j in range(8):
        g, r, te, tu, _ = b.step(acts[j])
        assert torch.equal(gk[j], g), (A, n, j)
        assert torch.equal(rk[j].view(torch.int64), r.view(torch.int64)) and torch.equal(tk[j], te) and torch.equal(uk[j], tu)
    assert torch.equal(a.state, b.state)
    g8 = c.step_k(8, actions=acts)[0]
    assert torch.equal(g8, b.obs) and torch.equal(c.state, b.state)
    # device-drawn actions: the keep-all steps draw the same stream as one K-step launch
    gk = a.step_k(8, action_step=100, keep_all=True)[0]
    g8 = c.step_k(8, action_step=100)[0]
    assert torch.equal(gk[-1], g8) and torch.equal(a.state, c.state)


def test_grid_observation_into_an_odd_byte_offset():
    for A in (1, 2):
        env = _coop(129, A, obs_spaces=None)      # feature-vector mode: grid_observation works there too
        env.reset()
        env.step(env.random_actions(0))
        shape = env._grid_shape
        size = int(np.prod(shape))
        buf = torch.full((size + 2,), 0xAB, dtype=torch.uint8, device="cuda")
        out = buf[1:1 + size].view(shape)
        assert out.data_ptr() % 2 == 1
        got = env.grid_observation(out=out)
        assert got.data_ptr() == out.data_ptr()
        assert int(buf[0]) == 0xAB and int(buf[-1]) == 0xAB
        _assert_grid(out, _own_grid(env), f"A={A} odd offset")
        assert torch.equal(env.grid_observation(), out)
        with pytest.raises(ValueError):
            env.grid_observation(out=torch.zeros(shape, dtype=torch.int32, device="cuda"))


# ---------------------------------------------------------------------------------------------------- 5. semantics
def test_grid_observe_masked_reset_auto_reset_and_cook():
    n = 257
    env = _coop(n, seed=5)
    twin = _coop(n, seed=5, obs_spaces=None)
    lids = env.default_layout_ids()
    env.reset(layout_ids=lids)
    twin.reset(layout_ids=lids)
    for s in range(10):                          # the device cook decides the same in both modes
        act, crashed = env.heuristic_actions()
        act2, crashed2 = twin.heuristic_actions()
        assert torch.equal(act, act2) and torch.equal(crashed, crashed2), s
        env.step(act.clone())
        twin.step(act2.clone())
        assert torch.equal(env.state, twin.state), s
    last = env.obs.clone()
    env.obs.fill_(0xFF)
    assert torch.equal(env.observe(), last)
    assert torch.equal(env.observe(), last)      # idempotent
    # a masked reset changes only the masked environments' grids
    mask = np.arange(n) % 3 == 0
    lids2 = (lids.cpu().numpy() + 1 + np.arange(n)) % env.tables.num_layouts
    fresh = _coop(n, seed=5)
    fresh_grid = fresh.reset(layout_ids=lids2).clone()
    after = env.reset(layout_ids=lids2, mask=mask)
    m = torch.from_numpy(mask).cuda()
    assert torch.equal(after[m], fresh_grid[m]) and torch.equal(after[~m], last[~m])
    # an auto-reset step shows the new episode: max_steps = 3 ends every episode at step 3
    ar = _coop(64, seed=9, auto_reset=True, max_steps=3)
    ar.reset()
    for s in range(3):
        ar.step(ar.random_actions(s))
    nxt = _coop(64, seed=9)
    want = nxt.reset(layout_ids=ar.default_layout_ids(episode=1))
    got = ar.step(ar.random_actions(3))[0]
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------------- 6. launches
_PROFILE_STEP = r"""
import json, sys
import torch
sys.path.insert(0, sys.argv[1])
from tests.test_gpu_grid import _coop
env = _coop(32768)
env.reset()
act = env.random_actions(0)
env.step(act)
torch.cuda.synchronize()
l0 = env.lib.cz_launch_count()
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    env.step(act)
    torch.cuda.synchronize()
names = sorted({e.key[e.key.index("cz_"):].split("(")[0] for e in prof.key_averages() if "cz_" in e.key})
print(json.dumps({"launches": env.lib.cz_launch_count() - l0, "kernels": names}))
"""


def test_large_grid_step_launches_dynamics_and_grid_kernels_only():
    """one in-place grid step of 32768 environments under torch.profiler: the dynamics-only kernel and the grid kernel.
    The profiler runs in a process of its own, so that this test leaves the profiler state of the test process as it was."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", _PROFILE_STEP, root], cwd=root, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    names = set(out["kernels"])
    assert out["launches"] == 2, out
    assert "cz_grid_kernel<2>" in names, names
    assert any(k.startswith("cz_env_kernel<0, 2, 2>") for k in names), names     # MODE_STEP, OBS_NONE (dynamics only), 2 agents
    assert not any("obs" in k or "warp" in k for k in names), names


# ---------------------------------------------------------------------------------------------------- 7. errors, wrappers
def test_grid_mode_errors():
    from cooking_zoo_b200 import BatchedCookingEnv
    from cooking_zoo_b200.mixed import MixedAgentCookingEnv
    with pytest.raises(NotImplementedError):
        _coop(8, obs_spaces=["grid", "feature_vector"])
    with pytest.raises(NotImplementedError):
        _coop(8, pipelined=True)
    with pytest.raises(ValueError):
        _coop(8, obs_dtype=torch.float32)
    with pytest.raises(NotImplementedError):
        MixedAgentCookingEnv([1, 2], "coop_test", "example", 400, RECIPES, obs_spaces=["grid"] * 2)
    env = _coop(8)
    assert isinstance(env, BatchedCookingEnv) and env.obs_mode == "grid"
    lib, h = env.lib, env._handle
    assert lib.cz_grid_channels(h) == 46 and lib.cz_grid_channels(None) == -1
    assert lib.cz_observe_grid(None, env.state.data_ptr(), env.obs.data_ptr(), 8, None) == -1
    assert lib.cz_observe_grid(h, None, env.obs.data_ptr(), 8, None) == -1
    assert lib.cz_observe_grid(h, env.state.data_ptr(), None, 8, None) == -1
    assert lib.cz_observe_grid(h, env.state.data_ptr(), env.obs.data_ptr(), 0, None) == 0


def test_parallel_env_grid_spaces():
    from cooking_zoo_b200.wrappers import parallel_env
    env = parallel_env(level="coop_test", meta_file="example", num_agents=2, max_steps=400, recipes=RECIPES,
                       obs_spaces=["grid"] * 2, end_condition_all_dishes=True, action_scheme="scheme3")
    space = env.observation_space("player_1")
    assert tuple(space.shape) == (46, 7, 7) and np.dtype(space.dtype) == np.uint8
    obs, _ = env.reset(options={"layout_id": 3})
    for i in range(2):
        assert obs[f"player_{i}"].dtype == np.uint8
        assert np.array_equal(obs[f"player_{i}"], env.backend.obs[0, i].cpu().numpy())
    obs, *_ = env.step({"player_0": 1, "player_1": 2})
    for i in range(2):
        assert np.array_equal(obs[f"player_{i}"], env.backend.obs[0, i].cpu().numpy())
    _assert_grid(env.backend.obs, _own_grid(env.backend), "parallel_env step")
