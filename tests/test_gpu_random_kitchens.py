"""GPU: every row writer and the device cook on random kitchens (tests/kitchens.py), against the oracles.

The fixed kitchens of the golden traces and of the exhaustive locksteps give only a handful of observation plans.  Random
kitchens vary what the row writers depend on: one or several computed ranges, table runs, one or two (observer, slot)
pairs per lane, odd row lengths, the parity of A * L, 16- or 32-lane warp groups.  Each kitchen here runs every path
the library can take for its plan (selected through the environment variables read when the tables are created) and
compares every environment at every step with oracle/cz_oracle.c (CBatch), which tests/test_random_kitchens.py holds
to the Python oracle on the same kitchens.  The device cook (cz_policy_act) is compared with oracle/cz_policy.py."""
import numpy as np
import pytest
import torch

from oracle import cz_policy
from oracle.cz_oracle import OracleEnv, SpawnStream
from tests.kitchens import DEVICE_KITCHENS, kitchen, kitchen_config, plan_class, served_recipes
from tests.replay import assert_state_equal

pytestmark = pytest.mark.gpu
N = 3001            # odd: the last block is ragged; >= 2 * ENVS_WARPS * SMs and below one wave of the warp kernel
N_LARGE = 20483     # above the default two-kernel threshold (CZ_TWO_KERNEL_MIN_ENVS = 20480)
STEPS = 40
ENVS_WARPS = 8
LARGE = [32, 1017, 68, 1011, 3, 9, 2]   # each class (packed with one and with several agents) at N_LARGE
TWO = {"CZ_WARP_MAX_ENVS": "0", "CZ_TWO_KERNEL_MIN_ENVS": "1"}
ARMS = {   # name: (environment variables, constructor arguments)
    "warp": ({}, {}),
    "warp32": ({"CZ_WARP_GROUP": "32"}, {}),
    "lane": ({"CZ_WARP_MAX_ENVS": "0"}, {}),
    "lane_stg": ({"CZ_WARP_MAX_ENVS": "0", "CZ_OBS_PATH": "stg"}, {}),
    "two": (TWO, {}),
    "round1": (dict(TWO, CZ_WHOLE_ROWS="0"), {}),
    "generic2": (dict(TWO, CZ_GENERIC="2"), {}),
    "generic1": (dict(TWO, CZ_GENERIC="1"), {}),
    "f32": ({}, {"obs_dtype": torch.float32}),
    "f32_one": ({"CZ_OBS32_PAIR": "0"}, {"obs_dtype": torch.float32}),
    "pipelined": ({}, {"pipelined": True}),
    "k8": ({}, {}),
}


def _kernels(prof):
    """names of the library's kernels a torch.profiler run saw, template arguments included"""
    out = set()
    for e in prof.key_averages():
        if "cz_" in e.key:
            out.add(e.key[e.key.index("cz_"):].split("(")[0])
    return out


def _launches(arm, cls):
    """launches of one step (of 8 steps for k8) where they identify the path; None: not asserted"""
    packed = cls.startswith("packed")
    if arm in ("warp", "warp32"):
        return 1                                    # warp kernel (packed) or the fused generic kernel
    if arm in ("lane", "lane_stg"):
        return 2 if cls == "packed64" else 1        # 33-64 pair plans always take dynamics + row writer
    if arm == "k8":
        return 1 if packed else 8
    if arm == "pipelined":
        return None
    return 2


def _make(lp, mp, cfg, seed, n, monkeypatch, env_vars=None, max_steps=STEPS, **kw):
    from cooking_zoo_b200 import BatchedCookingEnv
    for k, v in (env_vars or {}).items():
        monkeypatch.setenv(k, v)
    try:
        return BatchedCookingEnv(n, lp, mp, cfg["A"], max_steps, cfg["recipes"], end_condition_all_dishes=cfg["end_all"],
                                 action_scheme=cfg["scheme"], layout_pool_size=16, layout_seed=seed, seed=seed,
                                 **(cfg["spawn"] or {}), **kw)
    finally:
        for k in (env_vars or {}):
            monkeypatch.delenv(k)


def _cbatch(env, lids, cfg, seed):
    from oracle.cz_oracle_c import CBatch
    cpu = CBatch([env.tables.layouts[l] for l in lids], [cfg["recipes"]] * len(lids), STEPS,
                 end_condition_all_dishes=cfg["end_all"], action_scheme=cfg["scheme"], **(cfg["spawn"] or {}))
    if cfg["spawn"]:
        for k, e in enumerate(cpu.envs):
            cpu.lib.czo_set_stream(e.h, seed, k, 1)
    return cpu


def _first_bad(got, want, live, ctx):
    bad = (got != want)
    while bad.dim() > 1:
        bad = bad.any(-1)
    bad &= live
    if bool(bad.any()):
        raise AssertionError(f"{ctx}: environments {bad.nonzero().flatten()[:8].tolist()} differ")


def _lockstep(seed, arms, n, monkeypatch, tmp):
    """every arm of `arms` on kitchen `seed`, n environments, STEPS steps, every environment against CBatch"""
    lp, mp, _ = kitchen(seed, str(tmp))
    cfg = kitchen_config(seed)
    A = cfg["A"]
    envs = {a: _make(lp, mp, cfg, seed, n, monkeypatch, ARMS[a][0] if a in ARMS else {}, **(ARMS[a][1] if a in ARMS else {}))
            for a in arms}
    t = next(iter(envs.values())).tables
    cls = plan_class(t)
    if not cls.startswith("packed") and "pipelined" in envs:      # the pipelined step is for packed plans
        envs.pop("pipelined").close()
    lids = next(iter(envs.values())).default_layout_ids().cpu().numpy()
    cpu = _cbatch(envs[next(iter(envs))], lids, cfg, seed)
    want0 = torch.from_numpy(cpu.observe().copy()).cuda()
    for a, env in envs.items():
        o = env.reset(layout_ids=lids)
        w = want0.float().view(torch.int32) if env.obs_dtype == torch.float32 else want0.view(torch.int64)
        _first_bad(o.view(w.dtype), w, torch.ones(n, dtype=torch.bool, device="cuda"), f"kitchen {seed} {a} reset")
    rng = np.random.default_rng(seed)
    n_act = t.num_actions
    acts = np.zeros((STEPS, n, A), np.uint8)
    prev = np.zeros((n, A), np.uint8)
    for s in range(STEPS):
        prev = np.where(rng.random((n, A)) < 0.5, prev, rng.integers(0, n_act, size=(n, A))).astype(np.uint8)
        acts[s] = prev
    acts_d = torch.from_numpy(acts).cuda()
    live = torch.ones(n, dtype=torch.bool, device="cuda")     # episode not over before this step (no auto-reset here)
    k_out = None
    kernels = {}           # arm -> the library's kernels its first step launched (torch.profiler)
    for s in range(STEPS):
        outs = {}
        for a, env in envs.items():
            ctx = f"kitchen {seed} ({cls}, A={A}) arm {a} step {s}"
            l0 = env.lib.cz_launch_count()
            prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) if s == 0 else None
            if prof:
                prof.__enter__()
            if a == "k8":
                if s % 8 == 0:
                    k_out = env.step_k(8, actions=acts_d[s:s + 8], keep_all=True)
                    want = _launches(a, cls)
                    assert env.lib.cz_launch_count() - l0 == want, ctx
            else:
                o, r, te, tu, _ = env.step(acts_d[s])
                if a == "pipelined":
                    env.wait()
            if prof:
                torch.cuda.synchronize()
                prof.__exit__(None, None, None)
                kernels[a] = _kernels(prof)
            if a == "k8":
                outs[a] = tuple(x[s % 8] for x in k_out[:4])
                continue
            want = _launches(a, cls)
            if want is not None:
                assert env.lib.cz_launch_count() - l0 == want, ctx
            outs[a] = (o, r, te, tu)
        co, cr, cte, ctu = cpu.step(acts[s])
        ref_o = torch.from_numpy(co).cuda()
        ref_o32 = ref_o.float().view(torch.int32)
        ref_o = ref_o.view(torch.int64)
        ref_r = torch.from_numpy(cr).cuda().view(torch.int64)
        ref_te, ref_tu = torch.from_numpy(cte).cuda(), torch.from_numpy(ctu).cuda()
        ref_err = torch.tensor([e.error for e in cpu.envs], dtype=torch.int32, device="cuda")
        for a, (o, r, te, tu) in outs.items():
            ctx = f"kitchen {seed} ({cls}, A={A}) arm {a} step {s}"
            if o.dtype == torch.float32:
                _first_bad(o.view(torch.int32), ref_o32, live, ctx + " rows (f32)")
            else:
                _first_bad(o.view(torch.int64), ref_o, live, ctx + " rows")
            _first_bad(r.view(torch.int64), ref_r, live, ctx + " rewards")
            _first_bad(te, ref_te, live, ctx + " terminated")
            _first_bad(tu, ref_tu, live, ctx + " truncated")
            if a != "k8" or s % 8 == 7:
                _first_bad(envs[a].error_flags, ref_err, live, ctx + " error_flags")
        live &= ~ref_te.bool().any(1)
    assert int(live.sum()) > 0
    # observe() rewrites every row from the state (cz_observe's own dispatch)
    for a, env in envs.items():
        env.wait()
        last = k_out[0][-1].clone() if a == "k8" else env.obs.clone()
        env.obs.fill_(float("nan"))
        got = env.observe()
        w = torch.int32 if env.obs_dtype == torch.float32 else torch.int64
        assert torch.equal(got.view(w), last.view(w)), f"kitchen {seed} arm {a}: observe() != the last step's rows"
    # the state of 64 environments that ran to the end
    picks = np.random.default_rng(seed).choice(live.nonzero().flatten().cpu().numpy(), size=min(64, int(live.sum())),
                                               replace=False)
    for a, env in envs.items():
        states = env.export_state()
        for k in picks:
            assert_state_equal(cpu.envs[k].export_state(), states[k], f"kitchen {seed} arm {a} env {k}")
    # a masked reset of every third environment: fresh rows there, every other row unchanged
    mask = np.arange(n) % 3 == 0
    lids2 = (lids + 1 + np.arange(n)) % t.num_layouts
    fresh = _cbatch(envs[next(iter(envs))], lids2[mask], cfg, seed).observe()
    for a, env in envs.items():
        before = env.obs.clone()
        after = env.reset(layout_ids=lids2, mask=mask)
        env.wait()
        w = torch.int32 if env.obs_dtype == torch.float32 else torch.int64
        want = torch.from_numpy(fresh).cuda()
        want = want.float() if env.obs_dtype == torch.float32 else want
        m = torch.from_numpy(mask).cuda()
        assert torch.equal(after[m].view(w), want.view(w)), f"kitchen {seed} arm {a}: masked reset rows"
        assert torch.equal(after[~m].view(w), before[~m].view(w)), f"kitchen {seed} arm {a}: rows outside the mask changed"
    for env in envs.values():
        env.close()
    if cls.startswith("packed"):      # K steps in one launch, and single steps of this batch size, on the warp kernel
        for a in ("warp", "warp32", "k8"):
            if a in kernels:
                assert any(k.startswith("cz_warp_kernel") for k in kernels[a]), (seed, a, kernels[a])
    return cls, t, kernels


@pytest.mark.parametrize("seed", DEVICE_KITCHENS)
def test_every_path_against_the_compiled_oracle(seed, monkeypatch, tmp_path):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert 2 * ENVS_WARPS * sms <= N < sms * 28      # whole-row / single-pair writers engage; one wave of the warp kernel
    cls, t, kernels = _lockstep(seed, list(ARMS), N, monkeypatch, tmp_path)
    print(f"kitchen {seed}: {cls}, A={t.num_agents}, L={t.obs_len}, kernels launched "
          f"{sorted(set().union(*kernels.values()))}")


@pytest.mark.parametrize("seed", LARGE)
def test_default_dispatch_at_the_shipped_thresholds(seed, monkeypatch, tmp_path):
    cls, t, kernels = _lockstep(seed, ["default"], N_LARGE, monkeypatch, tmp_path)
    print(f"kitchen {seed}: {cls}, A={t.num_agents}, {N_LARGE} environments, kernels launched {sorted(kernels['default'])}")


def test_k_steps_keep_all_with_step_blocks_off_16_bytes(monkeypatch, tmp_path):
    """kitchen 0 (one agent, odd L) at an odd batch: outside the warp kernel, step k of a KEEP_ALL call writes its rows
    k * n * A * L elements into the buffer, which is not a multiple of 16 bytes (nor, in float32, of 4 elements).  Such
    calls used to be refused as misaligned ("obs must be 16-byte aligned") from the second step on."""
    lp, mp, _ = kitchen(0, str(tmp_path))
    cfg = kitchen_config(0)
    for dtype, w in ((torch.float64, torch.int64), (torch.float32, torch.int32)):
        a, b = (_make(lp, mp, cfg, 0, N, monkeypatch, obs_dtype=dtype) for _ in range(2))
        assert (N * cfg["A"] * a.obs_len * a.obs.element_size()) % 16 != 0
        a.reset(); b.reset()
        g = torch.Generator().manual_seed(5)
        acts = torch.randint(0, a.tables.num_actions, (8, N, cfg["A"]), generator=g, dtype=torch.uint8).cuda()
        obs, rew, te, tu, _ = a.step_k(8, actions=acts, keep_all=True)
        for k in range(8):
            o, r, te1, tu1, _ = b.step(acts[k])
            assert torch.equal(obs[k].view(w), o.view(w)) and torch.equal(rew[k].view(torch.int64), r.view(torch.int64)), k
            assert torch.equal(te[k], te1) and torch.equal(tu[k], tu1), k
        assert torch.equal(a.state, b.state)
        a.close(); b.close()


# ---- the device cook -----------------------------------------------------------------------------------------------
COOK_KITCHENS = [   # seed, options
    (32, {}), (16, {}), (29, {}), (28, {"generic": True}), (1, {}), (49, {}), (68, {}), (117, {}), (77, {}), (12, {}),
    (189, {}), (36, {"auto_reset": True}),
]
COOK_N, COOK_STEPS = 512, 60


def _decode(actions, crashed, A):
    """device (actions, crashed bits) -> the oracle's convention: -1 where the cook raised"""
    a = actions.cpu().numpy().astype(np.int64)
    c = crashed.cpu().numpy()
    for i in range(A):
        bad = (c >> i) & 1 == 1
        assert (a[bad, i] == 0).all()
        a[bad, i] = -1
    return a


def _cook_lockstep(seed, opts, monkeypatch, tmp):
    from cooking_zoo_b200.tables import ROW_EPISODE
    lp, mp, level = kitchen(seed, str(tmp))
    cfg = dict(kitchen_config(seed))
    A = cfg["A"]
    served = served_recipes(level)
    assert served, seed
    auto = bool(opts.get("auto_reset"))
    cfg["recipes"] = [served[i % len(served)] for i in range(A)]
    if auto:
        cfg["spawn"] = None
    max_steps = 25 if auto else 200
    env_vars = {"CZ_GENERIC": "1"} if opts.get("generic") else {}
    mk = lambda: _make(lp, mp, cfg, seed, COOK_N, monkeypatch, env_vars, max_steps=max_steps, recipe_pool=served,
                       auto_reset=auto)
    env, plain = mk(), mk()
    t = env.tables
    names = t.recipe_names
    rng = np.random.default_rng(seed)
    if auto:
        lids = env.default_layout_ids(episode=0).cpu().numpy()
        rids = np.tile(np.asarray(t.default_recipes, np.uint8), (COOK_N, 1))
        env.reset()
    else:
        lids = rng.integers(0, t.num_layouts, size=COOK_N).astype(np.int32)
        rids = rng.integers(0, len(served), size=(COOK_N, A)).astype(np.uint8)
        rids = np.array([[names.index(served[r]) for r in row] for row in rids], np.uint8)
        env.reset(layout_ids=lids, recipe_ids=rids)
    cooks = torch.from_numpy(rids[:, :A].copy()).cuda()

    def oracle(k, layout, episode):
        kw = {}
        if cfg["spawn"]:
            kw = dict(cfg["spawn"], spawn_stream=SpawnStream(seed, k, episode))
        return OracleEnv(t.layouts[layout], [names[r] for r in rids[k]], max_steps,
                         end_condition_all_dishes=cfg["end_all"], action_scheme=cfg["scheme"], **kw)
    oracles = {k: oracle(k, lids[k], 1) for k in range(COOK_N)}
    ep_row = t.num_dyn_slots + A + ROW_EPISODE
    episode = env.state[ep_row].cpu().numpy().copy()
    alive = set(oracles)
    counts = {}
    resets = 0
    for s in range(COOK_STEPS):
        act_t, crash_t = env.heuristic_actions()
        act_t, crash_t = act_t.clone(), crash_t.clone()
        got = _decode(act_t, crash_t, A)
        for k in sorted(alive):
            want = cz_policy.heuristic_actions(oracles[k], [names[r] for r in rids[k, :A]])
            assert got[k].tolist() == want, f"kitchen {seed} env {k} step {s}: oracle {want}, device {got[k].tolist()}"
            for w in want:
                counts[w] = counts.get(w, 0) + 1
        ea, ec = env.heuristic_actions(cooks)           # explicit cook recipes: the node marks re-evaluated from the graph
        assert torch.equal(ea, act_t) and torch.equal(ec, crash_t), f"kitchen {seed} step {s}: explicit cook tensor"
        plain.state.copy_(env.state)
        if s == 0:
            monkeypatch.setenv("CZ_POLICY_ENV_MARKS", "0")     # read when the policy handle is created (first call)
        pa, pc = plain.heuristic_actions()
        monkeypatch.delenv("CZ_POLICY_ENV_MARKS", raising=False)
        assert torch.equal(pa, act_t) and torch.equal(pc, crash_t), f"kitchen {seed} step {s}: CZ_POLICY_ENV_MARKS=0"
        act = np.where(rng.random((COOK_N, A)) < 0.15, rng.integers(0, 5, size=(COOK_N, A)), np.maximum(got, 0))
        act = act.astype(np.uint8)
        _, _, term, _, _ = env.step(torch.from_numpy(act))
        term = term.cpu().numpy()
        now = env.state[ep_row].cpu().numpy()
        if auto:
            new_ids = {}
            for k in np.flatnonzero(now != episode):
                c = int(now[k])
                if c not in new_ids:
                    new_ids[c] = env.default_layout_ids(episode=c - 1).cpu().numpy()
                oracles[k] = oracle(k, new_ids[c][k], c)
                resets += 1
            for k in np.flatnonzero(now == episode):
                oracles[k].step(act[k])
            episode = now.copy()
            continue
        for k in sorted(alive):
            _, te, _, _ = oracles[k].step(act[k])
            assert [int(v) for v in te] == list(term[k]), f"kitchen {seed} env {k} step {s}"
            if any(te):
                alive.discard(k)
    if auto:
        assert resets >= COOK_N, resets
    env.close(); plain.close()
    return counts


def test_device_cook_against_the_policy_oracle(monkeypatch, tmp_path):
    counts = {}
    for seed, opts in COOK_KITCHENS:
        for k, v in _cook_lockstep(seed, opts, monkeypatch, tmp_path).items():
            counts[k] = counts.get(k, 0) + v
    print("cook decisions:", dict(sorted(counts.items())))
    assert set(counts) == {-1, 0, 1, 2, 3, 4}
    assert 2 * counts[-1] < sum(counts.values())
