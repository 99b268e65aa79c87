"""GPU + reference: the CUDA kernels in lockstep with the LIVE, unmodified reference (oracle/_ref travels to the GPU box:
python -m oracle.make_ref).  Fixed levels and the random levels / meta files of the property test, both kernel families."""
import os
import random

import numpy as np
import pytest
import torch

from oracle.cz_oracle import RECIPES, SpawnStream
from tests.replay import assert_state_equal, assert_obs_equal, bits, ROOT
from tests.kitchens import _random_level, _random_meta
from tests.test_oracle_vs_reference import OPEN4, META4

pytestmark = [pytest.mark.gpu, pytest.mark.reference]
BOOK = list(RECIPES)


def _lockstep(level, meta, A, recipes, scheme, seeds, steps, spawn=None, max_steps=60, end_all=True):
    from cooking_zoo_b200 import BatchedCookingEnv
    from oracle.ref_harness import RefEnv
    n_act = 8 if scheme == "scheme1" else 5
    kw = {}
    refs = []
    for k, seed in enumerate(seeds):
        rkw = {}
        if spawn:
            rkw = dict(agent_respawn_rate=spawn[0], agent_despawn_rate=spawn[1], grace_period=spawn[2],
                       spawn_stream=SpawnStream(99, k, 1))
        refs.append(RefEnv(seed, level, meta, A, max_steps, recipes, end_condition_all_dishes=end_all, action_scheme=scheme, **rkw))
    if spawn:
        kw = dict(agent_respawn_rate=spawn[0], agent_despawn_rate=spawn[1], grace_period=spawn[2], seed=99)
    n = len(refs)
    env = BatchedCookingEnv(n, level, meta, A, max_steps, recipes, end_condition_all_dishes=end_all, action_scheme=scheme,
                            layouts=[r.layout() for r in refs], **kw)
    obs = env.reset(layout_ids=np.arange(n)).cpu().numpy()
    for k, r in enumerate(refs):
        assert_state_equal(r.export_state(), env.export_state(env=k), f"{os.path.basename(level)} env {k} reset")
        assert_obs_equal(r.observe_all(), obs[k], f"env {k} reset")
    rng = np.random.default_rng(seeds[0])
    alive = set(range(n))
    prev = np.zeros((n, A), np.int64)
    for t in range(steps):
        act = np.where(rng.random((n, A)) < 0.4, prev, rng.integers(0, n_act, size=(n, A)))
        prev = act
        obs, rew, term, trunc, _ = env.step(torch.from_numpy(act.astype(np.uint8)))
        obs, rew, term, trunc = obs.cpu().numpy(), rew.cpu().numpy(), term.cpu().numpy(), trunc.cpu().numpy()
        flags = env.error_flags.cpu().numpy()
        for k in sorted(alive):
            ctx = f"{os.path.basename(level)} env {k} step {t}"
            try:
                r = refs[k].step(act[k])
            except IndexError:          # Appendix C-9
                assert flags[k] == 16, ctx
                alive.discard(k)
                continue
            assert np.array_equal(bits(r[0]), bits(rew[k])), ctx
            assert list(r[1]) == list(term[k]) and list(r[2]) == list(trunc[k]), ctx
            assert_state_equal(refs[k].export_state(), env.export_state(env=k), ctx)
            assert_obs_equal(refs[k].observe_all(), obs[k], ctx)
            assert flags[k] == 0, ctx
            if r[1].any() or refs[k].env.t >= max_steps:
                alive.discard(k)
        if not alive:
            break
    env.close()


@pytest.mark.parametrize("kernel", ["warp", "lane"])
def test_device_vs_live_reference_fixed_levels(kernel, monkeypatch):
    if kernel == "lane":
        monkeypatch.setenv("CZ_WARP_MAX_ENVS", "0")
    for level in ("coop_test", "switch_test", "coexistence_test"):
        for scheme in ("scheme1", "scheme3"):
            _lockstep(level, "example", 2, ["TomatoLettuceSalad", "CarrotBanana"], scheme, [61, 62, 63], 60)
    for A in (1, 2, 3, 4):
        _lockstep(OPEN4, META4, A, ["TomatoLettuceSalad", "CarrotBanana", "TomatoSalad", "no_recipe"][:A], "scheme3",
                  [70 + A, 80 + A], 60, spawn=(0.25, 0.1 if A > 1 else 0.0, 2))


@pytest.mark.parametrize("kernel", ["warp", "lane"])
def test_device_vs_live_reference_random_levels_and_meta_files(kernel, monkeypatch, tmp_path):
    if kernel == "lane":
        monkeypatch.setenv("CZ_WARP_MAX_ENVS", "0")
    for seed in range(3000, 3016):
        rng = random.Random(seed)
        lp, mp = str(tmp_path / f"level_{seed}.json"), str(tmp_path / f"meta_{seed}.json")
        level = _random_level(rng, lp)
        _random_meta(rng, level, mp)
        A = rng.randint(1, 4)
        recipes = [BOOK[rng.randrange(8)] for _ in range(A)]
        _lockstep(lp, mp, A, recipes, rng.choice(["scheme1", "scheme3"]), [seed % 97, seed % 89 + 100], 50,
                  spawn=(0.3, 0.1, 1) if (seed & 1 and A > 1) else None, max_steps=50, end_all=bool(seed & 2))
