"""CPU: oracle/cz_policy.py (the scripted cook restated) against the raw CookingAgent decisions
recorded from the unmodified reference (tests/golden/policy_*.npz), plus the host-built
reachability / first-step tables the device policy reads."""
import glob
import os

import numpy as np
import pytest

from oracle.cz_oracle import OracleEnv, SpawnStream
from oracle import cz_policy
from tests.replay import GOLDEN_DIR, load_golden


def policy_files():
    return sorted(glob.glob(os.path.join(GOLDEN_DIR, "policy_*.npz")))


def oracle_env(cfg, layout, n):
    sp = cfg.get("spawn")
    kw = {} if not sp else dict(agent_respawn_rate=sp["respawn"], agent_despawn_rate=sp["despawn"],
                                grace_period=sp["grace"], spawn_stream=SpawnStream(sp["seed"], n, 1))
    return OracleEnv(layout, cfg["recipes"], cfg["max_steps"], reward_scheme=cfg["reward_scheme"],
                     end_condition_all_dishes=cfg["end_all"], action_scheme=cfg.get("action_scheme", "scheme3"), **kw)


@pytest.mark.parametrize("path", policy_files(), ids=lambda p: p.split("/")[-1][:-4])
def test_policy_oracle_matches_recorded_cook(path):
    g = load_golden(path)
    cfg = g["config"]
    names = cfg.get("policy_recipes", cfg["recipes"])
    seen = set()
    for n, layout in enumerate(g["layouts"]):
        env = oracle_env(cfg, layout, n)
        for t in range(int(g["length"][n])):
            got = cz_policy.heuristic_actions(env, names[:cfg["num_agents"]])
            want = g["policy"][n, t].tolist()
            assert got == want, f"{path} trace {n} step {t}: cook {want}, oracle {got}"
            seen.update(want)
            env.step(g["actions"][n, t])
    assert seen - {-1, 0}, "the traces must contain real decisions"


def test_policy_goldens_cover_crashes_and_all_moves():
    seen = set()
    for path in policy_files():
        seen.update(np.unique(load_golden(path)["policy"]).tolist())
    assert seen == {-1, 0, 1, 2, 3, 4}


@pytest.mark.parametrize("level,meta,agents", [("coop_test", "example", 2), ("switch_test", "example", 2),
                                               ("coexistence_test", "example", 2),
                                               ("tests/golden/levels/open4.json", "tests/golden/levels/meta4.json", 4),
                                               ("tests/golden/levels/tiny4.json", "tests/golden/levels/meta4.json", 4),
                                               # kitchen_<seed>: tests/kitchens.kitchen(seed), meta file included; seeds
                                               # 1, 5, 9 and 13 are split in two by an inner wall, 4 is a rich kitchen
                                               ("kitchen_1", None, 2), ("kitchen_5", None, 4), ("kitchen_9", None, 1),
                                               ("kitchen_13", None, 3), ("kitchen_2", None, 2), ("kitchen_7", None, 3),
                                               ("kitchen_4", None, 2)])
def test_policy_tables_match_the_queue_level_searches(level, meta, agents, tmp_path):
    """reach / first_step / lists of cooking_zoo_b200/policy.py == oracle.cz_policy.reachable / walk on every cell pair"""
    from cooking_zoo_b200.tables import compile_tables, ROW_VARIANT
    from cooking_zoo_b200.policy import compile_policy_tables
    from tests.kitchens import kitchen
    from tests.replay import ROOT
    if level.startswith("kitchen_"):
        level, meta, _ = kitchen(int(level[len("kitchen_"):]), str(tmp_path))
    path = lambda p: os.path.join(ROOT, p) if p.endswith(".json") else p
    t = compile_tables(path(level), path(meta), agents, 100, ["TomatoSalad"] * agents, layout_pool_size=24, layout_seed=5)
    p = compile_policy_tables(t)
    col = t.num_dyn_slots + t.num_agents + ROW_VARIANT
    done = set()
    for li, lay in enumerate(t.layouts):
        v = int(t.pool[li, col])
        if v in done:
            continue
        done.add(v)
        env = OracleEnv(lay, ["TomatoSalad"] * agents, 100)
        floor = cz_policy._floor(env)
        for name, objs in env.by_type.items():
            from cooking_zoo_b200.entities import entity
            et = entity(name)
            if et.kind == "static":
                n = int(p["list_len"][v, et.static_code])
                assert p["lists"][v, et.static_code, :n].tolist() == [o.y * 8 + o.x for o in objs]
        cells = [(x, y) for y in range(t.height) for x in range(t.width)]
        for a in cells:
            ia = a[1] * 8 + a[0]
            for b in cells:
                ib = b[1] * 8 + b[0]
                r = cz_policy.reachable(env, a, b, floor)
                assert bool(int(p["reach"][v, ia]) >> ib & 1) == r, (v, a, b)
                assert int(p["first_step"][v, ia, ib]) == cz_policy.walk(env, a, b, floor), (v, a, b)
                assert r == cz_policy.reachable(env, b, a, floor)          # the cook's cache assumes symmetry
    assert len(done) == t.num_variants
