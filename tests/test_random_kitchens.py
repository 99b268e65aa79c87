"""CPU: the two oracles (oracle/cz_oracle.py and the compiled oracle/cz_oracle.c) in lockstep on random kitchens.

Both are pinned to the reference by the golden traces on fixed kitchens; here they check each other where no trace
reaches: random and rich kitchens (tests/kitchens.py), kitchens split by an inner wall, random meta counts and order,
OPTIONAL objects, 1-4 agents, both action schemes, despawn / respawn.  The device kernels are checked against the
compiled oracle on the same kitchens (tests/test_gpu_random_kitchens.py), so an agreement here carries the Python
oracle's authority over to them."""
import numpy as np
import pytest

from oracle.cz_oracle import OracleEnv, SpawnStream
from oracle.cz_oracle_c import COracleEnv
from tests.kitchens import DEVICE_KITCHENS, kitchen, kitchen_config, plan_class, warp_group
from tests.replay import assert_state_equal, bits

SEEDS = range(200)
CHUNK = 25
STEPS = 40


def _oracle_pair(layout, cfg, seed, k, max_steps):
    envs = []
    for cls in (OracleEnv, COracleEnv):
        kw = dict(cfg["spawn"], spawn_stream=SpawnStream(seed, k, 1)) if cfg["spawn"] else {}
        envs.append(cls(layout, cfg["recipes"], max_steps, end_condition_all_dishes=cfg["end_all"],
                        action_scheme=cfg["scheme"], **kw))
    return envs


@pytest.mark.parametrize("first", range(SEEDS.start, SEEDS.stop, CHUNK))
def test_python_and_compiled_oracles_agree_on_random_kitchens(first, tmp_path):
    from cooking_zoo_b200.tables import compile_tables
    for seed in range(first, first + CHUNK):
        lp, mp, _ = kitchen(seed, str(tmp_path))
        cfg = kitchen_config(seed)
        t = compile_tables(lp, mp, cfg["A"], STEPS, cfg["recipes"], layout_pool_size=2, layout_seed=seed)
        n_act = 8 if cfg["scheme"] == "scheme1" else 5
        for k, layout in enumerate(t.layouts):
            po, co = _oracle_pair(layout, cfg, seed, k, STEPS)
            rng = np.random.default_rng(seed * 10 + k)
            prev = np.zeros(cfg["A"], np.int64)
            for step in range(STEPS):
                ctx = f"kitchen {seed} layout {k} step {step}"
                act = np.where(rng.random(cfg["A"]) < 0.5, prev, rng.integers(0, n_act, size=cfg["A"]))
                prev = act
                try:
                    r1, te1, tu1, _ = po.step(act)
                except Exception as e:        # the reference raises here too (e.g. time-up with a despawned agent)
                    co.step(act)
                    assert co.error != 0, f"{ctx}: the Python oracle raised {e!r}, the compiled oracle reports no error"
                    break
                r2, te2, tu2, _ = co.step(act)
                assert np.array_equal(bits(r1), bits(r2)), ctx
                assert [int(v) for v in te1] == te2.tolist() and [int(v) for v in tu1] == tu2.tolist(), ctx
                assert_state_equal(po.export_state(), co.export_state(), ctx)
                for i in range(cfg["A"]):
                    assert np.array_equal(bits(po.observe(i)), bits(co.observe(i))), f"{ctx} agent {i}"
                assert po.error == co.error, ctx
                if any(te1) or po.t >= STEPS:
                    break


def test_the_device_kitchens_cover_every_plan_class(tmp_path):
    """the kitchens of tests/test_gpu_random_kitchens.py must give every (plan class, agent count) the library has its
    own kernels for: the packed plans with <= 32 pairs for 1-4 agents (cz_env_kernel<., ., NA>, cz_warp_kernel<NA, .>,
    cz_obs_whole_kernel<NA, false>, cz_obs_envs_kernel<NA, false>, cz_obs_single_pair_kernel, the float32 writers), the
    33-64 pair plans for 2-4 agents (cz_obs_whole_kernel<NA, true> ...), both warp-group widths (the tests force 32-lane groups on the others), and tables outside the
    packed class with A * L even, A * L odd and odd L (the any-plan writers, the STG path of the fused generic kernel)"""
    from cooking_zoo_b200.tables import compile_tables
    seen, groups, spawn, schemes = set(), set(), set(), set()
    for seed in DEVICE_KITCHENS:
        lp, mp, _ = kitchen(seed, str(tmp_path))
        cfg = kitchen_config(seed)
        t = compile_tables(lp, mp, cfg["A"], 40, cfg["recipes"], layout_pool_size=16, layout_seed=seed)
        cls = plan_class(t)
        seen.add((cls, cfg["A"]))
        if cls.startswith("packed"):
            groups.add((cfg["A"], warp_group(t)))
        spawn.add(bool(cfg["spawn"]))
        schemes.add(cfg["scheme"])
    print("(class, agents):", sorted(seen), "\n(agents, warp group) of packed plans:", sorted(groups))
    need = {("packed32", a) for a in (1, 2, 3, 4)} | {("packed64", a) for a in (2, 3, 4)}
    assert need <= seen, sorted(need - seen)
    assert {c for c, _ in seen} == {"packed32", "packed64", "generic_AL_even", "generic_AL_odd", "generic_odd_L"}
    assert {g for _, g in groups} == {16, 32}
    assert spawn == {False, True} and schemes == {"scheme1", "scheme3"}
