"""oracle/cz_oracle.py (and the compiled oracle) in lockstep with the LIVE, unmodified reference — every level, both
action schemes, despawn / respawn, 1-4 agents, plus property tests over random meta counts and random open levels.
Runs wherever the reference is importable: /root/reference in the build container, the verbatim copy in oracle/_ref
(python -m oracle.make_ref) on the GPU box."""
import os
import random

import numpy as np
import pytest

from oracle.cz_oracle import OracleEnv, RECIPES, SpawnStream
from oracle.cz_oracle_c import COracleEnv
from tests.kitchens import _random_level, _random_meta
from tests.replay import assert_state_equal, assert_obs_equal, bits, ROOT

pytestmark = pytest.mark.reference
BOOK = list(RECIPES)
OPEN4 = os.path.join(ROOT, "tests/golden/levels/open4.json")
TINY4 = os.path.join(ROOT, "tests/golden/levels/tiny4.json")
META4 = os.path.join(ROOT, "tests/golden/levels/meta4.json")


def _lockstep(seed, level, A, recipes, max_steps, end_all, steps, policy_seed, meta="example", scheme="scheme3", spawn=None,
              reward_scheme=None, with_c=True):
    from oracle.ref_harness import RefEnv
    n_act = 8 if scheme == "scheme1" else 5
    kw_ref, kws = {}, [{}, {}]
    if spawn:
        kw_ref = dict(agent_respawn_rate=spawn[0], agent_despawn_rate=spawn[1], grace_period=spawn[2],
                      spawn_stream=SpawnStream(seed, 3, 1))
        kws = [dict(agent_respawn_rate=spawn[0], agent_despawn_rate=spawn[1], grace_period=spawn[2],
                    spawn_stream=SpawnStream(seed, 3, 1)) for _ in range(2)]
    ref = RefEnv(seed, level, meta, A, max_steps, recipes, end_condition_all_dishes=end_all, action_scheme=scheme,
                 reward_scheme=reward_scheme, **kw_ref)
    envs = [OracleEnv(ref.layout(), recipes, max_steps, end_condition_all_dishes=end_all, action_scheme=scheme,
                      reward_scheme=reward_scheme, **kws[0])]
    if with_c:
        envs.append(COracleEnv(ref.layout(), recipes, max_steps, end_condition_all_dishes=end_all, action_scheme=scheme,
                               reward_scheme=reward_scheme, **kws[1]))
    for orc in envs:
        assert_state_equal(ref.export_state(), orc.export_state(), f"seed {seed} reset")
    rng = np.random.default_rng(policy_seed)
    prev = np.zeros(A, np.int64)
    for t in range(steps):
        ctx = f"{os.path.basename(level)} seed {seed} step {t}"
        act = np.where(rng.random(A) < 0.4, prev, rng.integers(0, n_act, size=A))
        prev = act
        try:
            r1 = ref.step(act)
        except IndexError:           # Appendix C-9: the reference raises on time-up with a despawned agent
            assert spawn and t + 1 >= max_steps, ctx
            for orc in envs:
                orc.step(act)
                assert orc.error == 16, ctx
            return
        for orc in envs:
            r2 = orc.step(act)
            assert np.array_equal(bits(r1[0]), bits(r2[0])), ctx
            for a, b in zip(r1[1:], r2[1:]):
                assert list(a) == [int(v) for v in b], ctx
            assert_state_equal(ref.export_state(), orc.export_state(), ctx)
            assert_obs_equal(ref.observe_all(), np.stack([orc.observe(i) for i in range(A)]), ctx)
        if r1[1].any() or ref.env.t >= max_steps:
            break
    for orc in envs:
        assert orc.error == 0


@pytest.mark.parametrize("seed", range(8))
def test_live_lockstep_coop_test(seed):
    A = 1 + seed % 2
    recipes = [BOOK[(seed + k) % len(BOOK)] for k in range(A)]
    _lockstep(seed, "coop_test", A, recipes, 150, bool(seed & 2), 150, 77 + seed)


@pytest.mark.parametrize("level", ["coop_test", "switch_test", "coexistence_test"])
@pytest.mark.parametrize("scheme", ["scheme1", "scheme3"])
def test_live_lockstep_levels_and_schemes(level, scheme):
    for seed in range(20, 24):
        _lockstep(seed, level, 2, [BOOK[seed % 8], BOOK[(seed + 3) % 8]], 120, bool(seed & 1), 120, seed, scheme=scheme,
                  reward_scheme={"recipe_reward": 20, "max_time_penalty": -5, "recipe_penalty": -40,
                                 "recipe_node_reward": 0.5 * (seed % 3)})


@pytest.mark.parametrize("A", [1, 2, 3, 4])
@pytest.mark.parametrize("level", [OPEN4, TINY4])
def test_live_lockstep_one_to_four_agents_with_despawn_and_respawn(level, A):
    recipes = ["TomatoLettuceSalad", "CarrotBanana", "TomatoSalad", "no_recipe"][:A]
    for seed in range(40, 43):
        _lockstep(seed, level, A, recipes, 60, True, 60, seed, meta=META4, spawn=(0.25, 0.1 if A > 1 else 0.0, 2),
                  scheme="scheme1" if seed % 2 else "scheme3")


# ---- property tests: random meta counts, random open levels (at most 8x8), random action streams -------------------
def test_property_random_levels_and_meta_files(tmp_path):
    hyp = pytest.importorskip("hypothesis")
    from hypothesis import given, settings, strategies as st, HealthCheck

    @settings(max_examples=25, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
    @given(st.integers(0, 10 ** 6), st.integers(1, 4), st.sampled_from(["scheme1", "scheme3"]), st.booleans())
    def run(seed, A, scheme, spawn):
        rng = random.Random(seed)
        lp, mp = str(tmp_path / f"level_{seed}.json"), str(tmp_path / f"meta_{seed}.json")
        level = _random_level(rng, lp)
        _random_meta(rng, level, mp)
        recipes = [BOOK[rng.randrange(8)] for _ in range(A)]
        _lockstep(seed % 1000, lp, A, recipes, 50, bool(seed & 1), 50, seed, meta=mp, scheme=scheme,
                  spawn=(0.3, 0.1, 1) if spawn and A > 1 else None)
    run()
