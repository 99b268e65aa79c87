"""GPU: cz_step(k_steps) — K steps in one launch of the warp-per-environment kernel (csrc/cz_warp.cuh) must give,
step by step, the bits of K launches of the lane-per-environment kernels (which the golden traces and the exhaustive
lockstep tests pin to the reference)."""
import os

import numpy as np
import pytest
import torch

from tests.kitchens import _random_level, _random_meta, _rich_level
from tests.replay import ROOT

pytestmark = pytest.mark.gpu

R2 = ["TomatoLettuceSalad", "CarrotBanana"]
R4 = ["TomatoLettuceSalad", "CarrotBanana", "TomatoSalad", "no_recipe"]
OPEN4 = (os.path.join(ROOT, "tests/golden/levels/open4.json"), os.path.join(ROOT, "tests/golden/levels/meta4.json"))

CASES = {
    "cfg3_coop2": dict(n=4096, level="coop_test", meta="example", A=2, recipes=R2, max_steps=23),
    "coop1_any": dict(n=1000, level="coop_test", meta="example", A=1, recipes=R2[:1], max_steps=17, end_all=False),
    "scheme1": dict(n=2049, level="coop_test", meta="example", A=2, recipes=R2, max_steps=40, action_scheme="scheme1"),
    "spawn": dict(n=1500, level="coop_test", meta="example", A=2, recipes=R2, max_steps=30,
                  agent_respawn_rate=0.3, agent_despawn_rate=0.15, grace_period=2),
    "switch": dict(n=1024, level="switch_test", meta="example", A=2, recipes=R2, max_steps=50),
    "coexist": dict(n=1024, level="coexistence_test", meta="example", A=2, recipes=R2, max_steps=50),
    "open4_a3": dict(n=777, level=OPEN4[0], meta=OPEN4[1], A=3, recipes=R4[:3], max_steps=30),
    "open4_a4_spawn": dict(n=600, level=OPEN4[0], meta=OPEN4[1], A=4, recipes=R4, max_steps=30,
                           agent_respawn_rate=0.3, agent_despawn_rate=0.1, grace_period=1),
    "book_recipes": dict(n=2048, level="coop_test", meta="example", A=2, recipes=R2, max_steps=60, book=True,
                         reward_scheme={"recipe_reward": 20, "max_time_penalty": -5, "recipe_penalty": -40,
                                        "recipe_node_reward": 1.5}),
}
BOOK = ["TomatoSalad", "TomatoLettuceSalad", "CarrotBanana", "MashedCarrotBanana", "CucumberOnion", "AppleWatermelon",
        "TomatoLettuceOnionSalad", "no_recipe"]


def _make(case, **kw):
    from cooking_zoo_b200 import BatchedCookingEnv
    c = dict(CASES[case])
    n, book = c.pop("n"), c.pop("book", False)
    env = BatchedCookingEnv(n, c.pop("level"), c.pop("meta"), c.pop("A"), c.pop("max_steps"), c.pop("recipes"),
                            end_condition_all_dishes=c.pop("end_all", True),
                            action_scheme=c.pop("action_scheme", "scheme3"), layout_pool_size=48, layout_seed=4,
                            auto_reset=True, seed=21, recipe_pool=BOOK if book else None, **c, **kw)
    rid = None
    if book:
        rid = torch.randint(0, len(BOOK), (n, 2), generator=torch.Generator().manual_seed(1), dtype=torch.uint8)
    env.reset(recipe_ids=rid)
    return env


def _sticky_actions(K, n, A, n_act, seed):
    rng = np.random.default_rng(seed)
    out = np.zeros((K, n, A), np.uint8)
    prev = np.zeros((n, A), np.uint8)
    for k in range(K):
        prev = np.where(rng.random((n, A)) < 0.45, prev, rng.integers(0, n_act, size=(n, A))).astype(np.uint8)
        out[k] = prev
    return torch.from_numpy(out).cuda()


@pytest.mark.parametrize("group", ["auto", "32"])
@pytest.mark.parametrize("case", list(CASES))
def test_k_steps_in_one_launch_equal_k_single_steps(case, group, monkeypatch):
    """group: lanes per environment in the warp kernel — auto = 16 (two environments per warp) when the tables have at
    most 16 dynamic slots, 32 otherwise; "32" forces one environment per warp"""
    K, rounds = 16, 5           # 80 steps: several auto-resets at these max_steps
    monkeypatch.setenv("CZ_WARP_MAX_ENVS", "0")          # reference arm of this test: the lane-per-environment kernels
    lane = _make(case)
    monkeypatch.delenv("CZ_WARP_MAX_ENVS")
    if group == "32":
        if lane.tables.num_dyn_slots > 16:
            pytest.skip("already one environment per warp")
        monkeypatch.setenv("CZ_WARP_GROUP", "32")
    warp = _make(case)
    assert torch.equal(lane.state, warp.state) and torch.equal(lane.obs.view(torch.int64), warp.obs.view(torch.int64))
    n, A = lane.num_envs, lane.num_agents
    l0 = warp.lib.cz_launch_count()
    for rd in range(rounds):
        acts = _sticky_actions(K, n, A, lane.tables.num_actions, 100 + rd)
        obs, rew, term, trunc, _ = warp.step_k(K, actions=acts, keep_all=True)
        l1 = warp.lib.cz_launch_count()
        assert l1 - l0 == 1                                # ONE launch for the K steps
        for k in range(K):
            o, r, te, tr, _ = lane.step(acts[k])
            ctx = f"{case} round {rd} step {k}"
            assert torch.equal(r.view(torch.int64), rew[k].view(torch.int64)), ctx
            assert torch.equal(te, term[k]) and torch.equal(tr, trunc[k]), ctx
            bad = (o.view(torch.int64) != obs[k].view(torch.int64)).nonzero()
            assert bad.numel() == 0, (ctx, bad[:5].tolist())
        assert torch.equal(lane.state, warp.state), f"{case} round {rd}: state"
        l0 = warp.lib.cz_launch_count()
    assert torch.equal(lane.error_flags, warp.error_flags)
    if "spawn" not in case:
        assert int(warp.error_flags.abs().sum()) == 0
    assert int(warp.info()["t"].max()) <= lane.max_steps and int(warp.state[-1].max()) >= 2   # episodes restarted inside a launch


def test_k_steps_without_keep_all_leave_the_last_step_in_the_buffers():
    a, b = _make("cfg3_coop2"), _make("cfg3_coop2")
    acts = _sticky_actions(12, a.num_envs, 2, 5, 7)
    obs_all, rew_all, te_all, tr_all, _ = a.step_k(12, actions=acts, keep_all=True)
    obs, rew, te, tr, _ = b.step_k(12, actions=acts)
    assert obs.shape == (a.num_envs, 2, a.obs_len)
    assert torch.equal(obs.view(torch.int64), obs_all[-1].view(torch.int64))
    assert torch.equal(rew.view(torch.int64), rew_all[-1].view(torch.int64))
    assert torch.equal(te, te_all[-1]) and torch.equal(tr, tr_all[-1]) and torch.equal(a.state, b.state)


@pytest.mark.parametrize("case", ["cfg3_coop2", "scheme1"])
def test_device_generated_actions_inside_the_k_step_launch(case, monkeypatch):
    """actions=None: the kernel draws step j's actions from the counter stream of cz_random_actions at index
    action_step + j — the same rollout as random_actions(j) + step(j) on the lane kernels"""
    monkeypatch.setenv("CZ_WARP_MAX_ENVS", "0")
    lane = _make(case)
    monkeypatch.delenv("CZ_WARP_MAX_ENVS")
    warp = _make(case)
    K = 20
    for rd in range(3):
        obs, rew, term, trunc, _ = warp.step_k(K, action_step=1000 + rd * K, keep_all=True)
        for k in range(K):
            o, r, te, tr, _ = lane.step(lane.random_actions(1000 + rd * K + k))
            assert torch.equal(o.view(torch.int64), obs[k].view(torch.int64)), (rd, k)
            assert torch.equal(r.view(torch.int64), rew[k].view(torch.int64)) and torch.equal(te, term[k])
    assert torch.equal(lane.state, warp.state)


def test_k_steps_fall_back_to_per_step_launches_outside_the_specialised_class(monkeypatch):
    """generic tables (CZ_GENERIC=1) and float32 rows have no warp kernel: cz_step(k_steps) loops over the per-step
    kernels inside the library and must still honour actions [K][n][A], KEEP_ALL and device actions"""
    ref = _make("cfg3_coop2")
    monkeypatch.setenv("CZ_GENERIC", "1")
    gen = _make("cfg3_coop2")
    monkeypatch.delenv("CZ_GENERIC")
    acts = _sticky_actions(6, ref.num_envs, 2, 5, 3)
    l0 = gen.lib.cz_launch_count()
    og, rg, *_ = gen.step_k(6, actions=acts, keep_all=True)
    assert gen.lib.cz_launch_count() - l0 == 6
    orf, rr, *_ = ref.step_k(6, actions=acts, keep_all=True)
    assert torch.equal(og.view(torch.int64), orf.view(torch.int64)) and torch.equal(rg.view(torch.int64), rr.view(torch.int64))
    og, *_ = gen.step_k(5, action_step=9)
    orf, *_ = ref.step_k(5, action_step=9)
    assert torch.equal(og.view(torch.int64), orf.view(torch.int64)) and torch.equal(gen.state, ref.state)
    f32 = _make("cfg3_coop2", obs_dtype=torch.float32)
    o32, *_ = f32.step_k(6, actions=acts, keep_all=True)
    o32b, *_ = f32.step_k(5, action_step=9)
    assert o32.shape == (6, ref.num_envs, 2, ref.obs_len) and o32.dtype == torch.float32
    assert torch.equal(o32b.view(torch.int32), orf.float().view(torch.int32)) and torch.equal(f32.state, ref.state)


def test_single_steps_of_small_batches_take_the_warp_kernel_and_ragged_sizes_work(monkeypatch):
    from cooking_zoo_b200 import BatchedCookingEnv
    for n in (1, 3, 5, 130):
        monkeypatch.setenv("CZ_WARP_MAX_ENVS", "0")
        lane = BatchedCookingEnv(n, "coop_test", "example", 2, 9, R2, action_scheme="scheme3", layout_pool_size=8,
                                 auto_reset=True, seed=2)
        monkeypatch.delenv("CZ_WARP_MAX_ENVS")
        warp = BatchedCookingEnv(n, "coop_test", "example", 2, 9, R2, action_scheme="scheme3", layout_pool_size=8,
                                 auto_reset=True, seed=2)
        lane.reset(); warp.reset()
        rng = np.random.default_rng(n)
        for t in range(30):
            act = torch.from_numpy(rng.integers(0, 5, size=(n, 2)).astype(np.uint8)).cuda()
            ol, rl, tl, ul, _ = lane.step(act)
            ow, rw, tw, uw, _ = warp.step(act)
            assert torch.equal(ol.view(torch.int64), ow.view(torch.int64)), (n, t)
            assert torch.equal(rl.view(torch.int64), rw.view(torch.int64)) and torch.equal(tl, tw) and torch.equal(ul, uw)
        assert torch.equal(lane.state, warp.state)


def test_k_steps_on_random_levels_and_meta_files(tmp_path, monkeypatch):
    """the property-test generator of tests/test_oracle_vs_reference.py (random open kitchens up to 8x8, random meta
    counts and order, OPTIONAL objects, 1-4 agents, both action schemes, despawn / respawn): K steps in one launch of the
    warp kernel against K launches of the lane kernels, table classes and group widths as they fall"""
    import random
    from cooking_zoo_b200 import BatchedCookingEnv
    widths = set()
    for seed in range(5000, 5024):
        rng = random.Random(seed)
        lp, mp = str(tmp_path / f"level_{seed}.json"), str(tmp_path / f"meta_{seed}.json")
        if seed % 3 == 0:
            level = _random_level(rng, lp)
            _random_meta(rng, level, mp)
            A = rng.randint(1, 4)
        else:
            _rich_level(rng, lp, mp)
            A = rng.randint(1, 2)           # 3-4 agents x ~25 computed slots would leave the packed class
        recipes = [BOOK[rng.randrange(8)] for _ in range(A)]
        scheme = rng.choice(["scheme1", "scheme3"])
        kw = dict(agent_respawn_rate=0.3, agent_despawn_rate=0.1, grace_period=1) if (seed & 1 and A > 1) else {}

        def make():
            e = BatchedCookingEnv(700, lp, mp, A, 25, recipes, end_condition_all_dishes=bool(seed & 2), action_scheme=scheme,
                                  layout_pool_size=40, layout_seed=seed, auto_reset=True, seed=seed, **kw)
            e.reset()
            return e
        monkeypatch.setenv("CZ_WARP_MAX_ENVS", "0")
        lane = make()
        monkeypatch.delenv("CZ_WARP_MAX_ENVS")
        warp = make()
        tb = warp.tables
        if tb.num_agents * tb.num_comp_slots <= 64 and tb.num_obs_ranges == 1 and tb.obs_table_len <= 128 and tb.obs_len % 2 == 0:
            widths.add(16 if lane.tables.num_dyn_slots <= 16 else 32)     # the warp kernel really ran
        n_act = lane.tables.num_actions
        for rd in range(3):
            acts = _sticky_actions(12, 700, A, n_act, seed + rd)
            obs, rew, term, trunc, _ = warp.step_k(12, actions=acts, keep_all=True)
            for k in range(12):
                o, r, te, tr, _ = lane.step(acts[k])
                ctx = (seed, rd, k)
                assert torch.equal(o.view(torch.int64), obs[k].view(torch.int64)), ctx
                assert torch.equal(r.view(torch.int64), rew[k].view(torch.int64)), ctx
                assert torch.equal(te, term[k]) and torch.equal(tr, trunc[k]), ctx
            assert torch.equal(lane.state, warp.state) and torch.equal(lane.error_flags, warp.error_flags), (seed, rd)
        lane.close(); warp.close()
    assert widths == {16, 32}
