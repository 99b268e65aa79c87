"""GPU: the CUDA path (through the C ABI) against the golden traces and the oracle."""
import numpy as np
import pytest
import torch

from oracle.cz_oracle import OracleEnv
from tests.replay import golden_files, load_golden, assert_state_equal, assert_obs_equal, bits, STATE_KEYS, package_recipes

pytestmark = pytest.mark.gpu


def _make(n, cfg, **kw):
    from cooking_zoo_b200 import BatchedCookingEnv
    sp = cfg.get("spawn")
    if sp:   # trace k is environment k of the shared spawn stream (episode 1 = after the first reset)
        kw = dict(kw, agent_respawn_rate=sp["respawn"], agent_despawn_rate=sp["despawn"], grace_period=sp["grace"],
                  seed=sp["seed"])
    return BatchedCookingEnv(n, cfg["level"], cfg["meta_file"], cfg["num_agents"], cfg["max_steps"],
                             cfg["recipes"], end_condition_all_dishes=cfg["end_all"],
                             reward_scheme=cfg["reward_scheme"], action_scheme=cfg.get("action_scheme", "scheme3"), **kw)


@pytest.mark.parametrize("kernel", ["warp", "lane"])
@pytest.mark.parametrize("path", golden_files(), ids=lambda p: p.split("/")[-1][:-4])
def test_cuda_replays_golden(path, kernel, monkeypatch):
    """Lockstep replay of traces recorded from the unmodified reference: bit-exact state,
    rewards (f64), flags and feature-vector observations (f64).  Small batches step on the
    warp-per-environment kernel (csrc/cz_warp.cuh); "lane" forces the lane-per-environment kernels
    (CZ_WARP_MAX_ENVS is read when the tables are created)."""
    if kernel == "lane":
        monkeypatch.setenv("CZ_WARP_MAX_ENVS", "0")
    g = load_golden(path)
    cfg = g["config"]
    n, A = len(g["layouts"]), cfg["num_agents"]
    with package_recipes(cfg):          # recipes registered through register_recipe (custom_recipes*.npz)
        env = _make(n, cfg, layouts=g["layouts"])
    obs = env.reset(layout_ids=np.arange(n)).cpu().numpy()
    states = env.export_state()
    for k in range(n):
        assert_state_equal({key: g[key][k, 0] for key in STATE_KEYS}, states[k], f"{path} trace {k} reset")
        assert_obs_equal(g["obs"][k, 0], obs[k], f"{path} trace {k} reset")
    T = g["actions"].shape[1]
    for t in range(T):
        live = [k for k in range(n) if t < g["length"][k]]
        if not live:
            break
        for k in live:
            for i in range(A):
                if g["teleport"][k, t, i, 0] >= 0:
                    env.teleport(k, i, *map(int, g["teleport"][k, t, i]))
        obs, rew, term, trunc, _ = env.step(torch.from_numpy(g["actions"][:, t].astype(np.uint8)))
        obs, rew, term, trunc = obs.cpu().numpy(), rew.cpu().numpy(), term.cpu().numpy(), trunc.cpu().numpy()
        states = env.export_state()
        for k in live:
            ctx = f"{path} trace {k} step {t}"
            assert np.array_equal(bits(g["reward"][k, t]), bits(rew[k])), ctx
            assert np.array_equal(g["term"][k, t], term[k]), ctx
            assert np.array_equal(g["trunc"][k, t], trunc[k]), ctx
            assert_state_equal({key: g[key][k, t + 1] for key in STATE_KEYS}, states[k], ctx)
            assert_obs_equal(g["obs"][k, t + 1], obs[k], ctx)
    # traces that end where the reference itself raised (Appendix C-9 fixtures) keep stepping past that point here and
    # are flagged, as they must be (tests/test_error_contract.py); every other trace stays clean
    clean = torch.from_numpy(np.asarray(g.get("raised", -np.ones(n)), np.int64) < 0).cuda()
    assert int(env.error_flags[clean].abs().sum()) == 0


def _oracle_lockstep(n_envs, check, steps, A, recipes, seed, max_steps=400, end_all=True, level="coop_test", meta="example"):
    cfg = dict(level=level, meta_file=meta, num_agents=A, max_steps=max_steps, recipes=recipes,
               end_all=end_all, reward_scheme=None)
    env = _make(n_envs, cfg, layout_pool_size=64, layout_seed=seed)
    lids = np.random.default_rng(seed).integers(0, 64, size=n_envs).astype(np.int32)
    obs = env.reset(layout_ids=lids).cpu().numpy()
    picks = np.linspace(0, n_envs - 1, check).astype(int)
    oracles = {int(k): OracleEnv(env.tables.layouts[lids[k]], recipes, max_steps, end_condition_all_dishes=end_all)
               for k in picks}
    for k, orc in oracles.items():
        assert_obs_equal(np.stack([orc.observe(i) for i in range(A)]), obs[k], f"env {k} reset")
    rng = np.random.default_rng(seed + 1)
    prev = np.zeros((n_envs, A), np.uint8)
    alive = set(oracles)
    for t in range(steps):
        act = np.where(rng.random((n_envs, A)) < 0.4, prev, rng.integers(0, 5, size=(n_envs, A))).astype(np.uint8)
        prev = act
        obs, rew, term, trunc, _ = env.step(torch.from_numpy(act))
        obs, rew, term, trunc = obs.cpu().numpy(), rew.cpu().numpy(), term.cpu().numpy(), trunc.cpu().numpy()
        st = env.state.cpu()
        for k in sorted(alive):
            orc = oracles[k]
            ctx = f"env {k} step {t}"
            r, te, tu, _ = orc.step(act[k])
            assert np.array_equal(bits(r), bits(rew[k])), ctx
            assert [int(v) for v in te] == list(term[k]) and [int(v) for v in tu] == list(trunc[k]), ctx
            assert_obs_equal(np.stack([orc.observe(i) for i in range(A)]), obs[k], ctx)
            if t % 16 == 0 or any(te) or any(tu):
                assert_state_equal(orc.export_state(), env.export_state(env=k), ctx)
            if any(te) or any(tu):
                alive.discard(k)
    return env


def test_cuda_vs_oracle_4096_envs():
    """BASELINE config 3 shape (4096 two-agent coop_test envs): 96 sampled envs in lockstep with the oracle."""
    _oracle_lockstep(4096, 96, 120, 2, ["TomatoLettuceSalad", "CarrotBanana"], seed=5)


def test_cuda_vs_oracle_per_layout_scan_orders():
    """a level whose OPTIONAL first Tomato entry can move the type behind the others: layouts disagree on the scan
    order of get_objects_at, so every layout keeps its own (tests/golden/levels/interleaved_optional.json)"""
    import os
    from tests.replay import ROOT
    env = _oracle_lockstep(2048, 64, 120, 2, ["TomatoLettuceSalad", "CarrotBanana"], seed=12,
                           level=os.path.join(ROOT, "tests/golden/levels/interleaved_optional.json"))
    assert len({s.tobytes() for s in env.tables.scan_order}) > 1


def test_cuda_vs_oracle_ragged_batch():
    """batch sizes that do not fill a warp / a block, single agent"""
    for n in (1, 31, 33, 129):
        _oracle_lockstep(n, min(n, 8), 40, 1, ["TomatoLettuceSalad"], seed=n, end_all=False)


def test_observe_is_idempotent_and_matches_step_obs():
    cfg = dict(level="coop_test", meta_file="example", num_agents=2, max_steps=400,
               recipes=["TomatoLettuceSalad", "CarrotBanana"], end_all=True, reward_scheme=None)
    env = _make(20000, cfg)
    env.reset()
    rng = np.random.default_rng(0)
    for t in range(30):
        obs, *_ = env.step(torch.from_numpy(rng.integers(0, 5, size=(20000, 2)).astype(np.uint8)))
    a = obs.clone()
    b = env.observe().clone()
    assert torch.equal(a.view(torch.int64), b.view(torch.int64))


def test_auto_reset_and_shard_independence():
    """truncation -> next step re-initialises from the pool draw cz_layout_draw(seed, env, episode);
    results do not depend on how the env range is split across devices/processes."""
    cfg = dict(level="coop_test", meta_file="example", num_agents=2, max_steps=7,
               recipes=["TomatoLettuceSalad", "CarrotBanana"], end_all=True, reward_scheme=None)
    n = 300
    whole = _make(n, cfg, auto_reset=True, seed=11, layout_pool_size=32)
    lo = _make(100, cfg, auto_reset=True, seed=11, layout_pool_size=32)
    hi = _make(200, cfg, auto_reset=True, seed=11, layout_pool_size=32, env_offset=100)
    for e in (whole, lo, hi):
        e.reset()
    rng = np.random.default_rng(3)
    P = whole.tables.num_layouts
    for t in range(20):
        act = rng.integers(0, 5, size=(n, 2)).astype(np.uint8)
        o, r, te, tr, info = whole.step(torch.from_numpy(act))
        o1, r1, te1, tr1, _ = lo.step(torch.from_numpy(act[:100]))
        o2, r2, te2, tr2, _ = hi.step(torch.from_numpy(act[100:]))
        assert torch.equal(o.view(torch.int64), torch.cat([o1, o2]).view(torch.int64))
        assert torch.equal(r.view(torch.int64), torch.cat([r1, r2]).view(torch.int64))
        assert torch.equal(tr, torch.cat([tr1, tr2])) and torch.equal(te, torch.cat([te1, te2]))
        tt = info["t"].cpu().numpy()
        if t % 8 == 6:      # step 7, 15: every env truncates
            assert tr.all() and (tt == 7).all()
        if t % 8 == 7:      # the step after: reset obs, zero reward, t == 0
            assert not tr.any() and (tt == 0).all() and float(r.abs().sum()) == 0.0
            episode = t // 8 + 1
            for k in (0, 57, 299):
                lid = whole.lib.cz_layout_draw(11, k, episode) % P
                orc = OracleEnv(whole.tables.layouts[lid], cfg["recipes"], 7, end_condition_all_dishes=True)
                assert_obs_equal(np.stack([orc.observe(i) for i in range(2)]), o[k].cpu().numpy(), f"autoreset env {k}")


@pytest.mark.parametrize("ring", [(2, 0), (3, 2), (4, 1)], ids=["pingpong", "ring3_bg2", "ring4_bg1"])
@pytest.mark.parametrize("level,agents", [("coop_test", 2), ("switch_test", 2), ("coexistence_test", 2),
                                          ("open4", 3), ("open4", 4)])
def test_pipelined_step_is_bit_identical_to_the_in_place_step(level, agents, ring):
    """throughput mode (cz_step_pipelined: two streams, a ring of state matrices) does the same work as cz_step;
    switch_test adds live Switch / Block slots to the observation writer, coexistence_test 16 static variants,
    the open kitchen with 3-4 agents the two-pairs-per-lane writer.  ring = (state matrices, dynamics blocks per SM):
    with a small dynamics grid the kernel loops over its tiles in the background of the row writer (cz_pipeline_config)"""
    import os
    from tests.replay import ROOT
    cfg = dict(level=level, meta_file="example", num_agents=agents, max_steps=30,
               recipes=["TomatoLettuceSalad", "CarrotBanana", "TomatoSalad", "no_recipe"][:agents], end_all=True,
               reward_scheme=None)
    if level == "open4":
        cfg.update(level=os.path.join(ROOT, "tests/golden/levels/open4.json"),
                   meta_file=os.path.join(ROOT, "tests/golden/levels/meta4.json"))
    n = 5000 if ring[1] == 0 else 50011          # the capped grid only differs from the full one on a large batch
    a = _make(n, cfg, auto_reset=True, seed=3, layout_pool_size=64)
    b = _make(n, cfg, auto_reset=True, seed=3, layout_pool_size=64, pipelined=True, pipeline_buffers=ring[0],
              background_dynamics=ring[1])
    a.reset(); b.reset()
    rng = np.random.default_rng(1)
    for t in range(70):
        act = torch.from_numpy(rng.integers(0, 5, size=(n, agents)).astype(np.uint8)).cuda()
        oa, ra, ta, ua, _ = a.step(act)
        ob, rb, tb, ub, _ = b.step(act)
        if t % 7 == 0 or t > 60:
            b.wait()
            torch.cuda.synchronize()
            assert torch.equal(oa.view(torch.int64), ob.view(torch.int64)), t
            assert torch.equal(ra.view(torch.int64), rb.view(torch.int64)) and torch.equal(ta, tb) and torch.equal(ua, ub)
            assert torch.equal(a.state, b.state)


@pytest.mark.parametrize("agents", [2, 4])
def test_masked_reset_touches_only_the_selected_environments(agents):
    """reset(mask=...) re-initialises state and rows of the masked environments only (2 agents: packed plan,
    4 agents: the 33-64 pair plan, whose masked reset runs on the generic kernel)"""
    import os
    from tests.replay import ROOT
    cfg = dict(level=os.path.join(ROOT, "tests/golden/levels/open4.json"),
               meta_file=os.path.join(ROOT, "tests/golden/levels/meta4.json"), num_agents=agents, max_steps=100,
               recipes=["TomatoLettuceSalad", "CarrotBanana", "TomatoSalad", "no_recipe"][:agents], end_all=True,
               reward_scheme=None)
    n = 777
    env = _make(n, cfg, layout_pool_size=32)
    fresh = env.reset().clone()
    first_state = env.state.clone()
    rng = np.random.default_rng(4)
    for t in range(25):
        env.step(torch.from_numpy(rng.integers(0, 5, size=(n, agents)).astype(np.uint8)))
    moved_obs, moved_state = env.obs.clone(), env.state.clone()
    mask = torch.from_numpy(rng.random(n) < 0.4)
    env.reset(layout_ids=env.default_layout_ids(0), mask=mask)
    m = mask.cuda()
    assert torch.equal(env.obs[m].view(torch.int64), fresh[m].view(torch.int64))
    assert torch.equal(env.obs[~m].view(torch.int64), moved_obs[~m].view(torch.int64))
    # episode counters differ after a second reset: compare everything but the EPISODE row
    assert torch.equal(env.state[:-1, m], first_state[:-1, m]) and torch.equal(env.state[:, ~m], moved_state[:, ~m])


def test_large_batch_two_kernel_step_equals_the_fused_kernel_on_a_ragged_batch(monkeypatch):
    """in-place steps of >= 20480 environments run the dynamics kernel and then the row-writer kernel; the fused kernel
    (forced here through CZ_TWO_KERNEL_MIN_ENVS=0, read when the tables are created) must give the same bits.
    50001 environments: neither a whole tile nor a whole writer block at the end."""
    cfg = dict(level="coop_test", meta_file="example", num_agents=2, max_steps=40,
               recipes=["TomatoLettuceSalad", "CarrotBanana"], end_all=True, reward_scheme=None)
    n = 50001
    a = _make(n, cfg, auto_reset=True, seed=8, layout_pool_size=64)
    monkeypatch.setenv("CZ_TWO_KERNEL_MIN_ENVS", "0")
    b = _make(n, cfg, auto_reset=True, seed=8, layout_pool_size=64)
    monkeypatch.delenv("CZ_TWO_KERNEL_MIN_ENVS")
    oa, ob = a.reset(), b.reset()
    assert torch.equal(oa.view(torch.int64), ob.view(torch.int64))
    rng = np.random.default_rng(2)
    l0 = a.lib.cz_launch_count()
    for t in range(45):
        act = torch.from_numpy(rng.integers(0, 5, size=(n, 2)).astype(np.uint8)).cuda()
        oa, ra, ta, ua, _ = a.step(act)
        l1 = a.lib.cz_launch_count()
        ob, rb, tb, ub, _ = b.step(act)
        l2 = a.lib.cz_launch_count()
        assert (l1 - l0, l2 - l1) == (2, 1)          # two kernels vs one fused kernel
        l0 = l2
        assert torch.equal(oa.view(torch.int64), ob.view(torch.int64)), t
        assert torch.equal(ra.view(torch.int64), rb.view(torch.int64)) and torch.equal(ta, tb) and torch.equal(ua, ub)
    assert torch.equal(a.state, b.state)


def test_pipelined_masked_reset_after_an_odd_number_of_steps_and_staged_actions():
    """ADVICE r01: a masked reset in pipelined mode must land in the ping-pong half that holds the current state and must
    not race the internal streams; host-side (numpy) actions go through the staging buffer, which a running dynamics kernel
    may still be reading unless the caller's stream trails it.  Compared step by step with the in-place environment."""
    cfg = dict(level="coop_test", meta_file="example", num_agents=2, max_steps=50,
               recipes=["TomatoLettuceSalad", "CarrotBanana"], end_all=True, reward_scheme=None)
    n = 20011
    a = _make(n, cfg, seed=3, layout_pool_size=64)
    b = _make(n, cfg, seed=3, layout_pool_size=64, pipelined=True)
    a.reset(); b.reset()
    rng = np.random.default_rng(5)

    def both(act):
        oa, ra, ta, ua, _ = a.step(act)
        ob, rb, tb, ub, _ = b.step(act)
        b.wait()
        assert torch.equal(oa.view(torch.int64), ob.view(torch.int64))
        assert torch.equal(ra.view(torch.int64), rb.view(torch.int64)) and torch.equal(ta, tb) and torch.equal(ua, ub)
        assert torch.equal(a.state, b.state)

    for t in range(3):                                    # odd: the current state sits in the second half
        both(rng.integers(0, 5, size=(n, 2)).astype(np.uint8))            # numpy actions -> staging buffer
    mask = torch.from_numpy(rng.random(n) < 0.3)
    lids = a.default_layout_ids(1)
    oa = a.reset(layout_ids=lids, mask=mask)
    ob = b.reset(layout_ids=lids, mask=mask)
    assert torch.equal(oa.view(torch.int64), ob.view(torch.int64)) and torch.equal(a.state, b.state)
    for t in range(4):
        both(rng.integers(0, 5, size=(n, 2)).astype(np.uint8))
    a.reset(); b.reset()                                  # full reset after an even + odd mix
    for t in range(3):
        both(torch.from_numpy(rng.integers(0, 5, size=(n, 2)).astype(np.uint8)).cuda())
    # back-to-back pipelined steps from host arrays with no wait in between: the staging copy of step k+1 is ordered after
    # the dynamics of step k (cz_step_pipelined makes the caller's stream trail them)
    acts = [rng.integers(0, 5, size=(n, 2)).astype(np.uint8) for _ in range(6)]
    for act in acts:
        b.step(act)
    b.wait()
    for act in acts:
        a.step(act)
    assert torch.equal(a.state, b.state) and torch.equal(a.obs.view(torch.int64), b.obs.view(torch.int64))


@pytest.mark.parametrize("split", ["2", "3", "8"])
def test_split_in_place_step_equals_the_unsplit_step(split, monkeypatch):
    """in-place steps of >= 98304 environments run as column ranges (dynamics of range c+1 under the rows of range c,
    csrc cz_step_split); CZ_SPLIT=1 is the plain two-launch step.  100001 environments: ragged last range."""
    cfg = dict(level="coop_test", meta_file="example", num_agents=2, max_steps=30,
               recipes=["TomatoLettuceSalad", "CarrotBanana"], end_all=True, reward_scheme=None)
    n = 100001
    monkeypatch.setenv("CZ_SPLIT", "1")
    a = _make(n, cfg, auto_reset=True, seed=8, layout_pool_size=64)
    monkeypatch.setenv("CZ_SPLIT", split)
    b = _make(n, cfg, auto_reset=True, seed=8, layout_pool_size=64)
    a.reset(); b.reset()
    rng = np.random.default_rng(2)
    for t in range(35):
        act = torch.from_numpy(rng.integers(0, 5, size=(n, 2)).astype(np.uint8)).cuda()
        l0 = a.lib.cz_launch_count()
        oa, ra, ta, ua, _ = a.step(act)
        l1 = a.lib.cz_launch_count()
        ob, rb, tb, ub, _ = b.step(act)
        l2 = a.lib.cz_launch_count()
        assert l1 - l0 == 2 and l2 - l1 == 2 * min(int(split), -(-n // (((-(-n // int(split))) + 255) & ~255)))
        assert torch.equal(oa.view(torch.int64), ob.view(torch.int64)), t
        assert torch.equal(ra.view(torch.int64), rb.view(torch.int64)) and torch.equal(ta, tb) and torch.equal(ua, ub)
    assert torch.equal(a.state, b.state) and torch.equal(a.error_flags, b.error_flags)


def test_device_action_stream_matches_its_definition_and_is_shard_independent():
    """cz_random_actions: floor(cz_spawn_uniform(seed ^ 0xA5.., env, 0, step, agent) * len(ACTIONS)); scheme1 draws from 8
    actions, scheme3 from 5; the stream of an environment does not depend on the shard it lives in"""
    cfg = dict(level="coop_test", meta_file="example", num_agents=2, max_steps=50,
               recipes=["TomatoLettuceSalad", "CarrotBanana"], end_all=True, reward_scheme=None)
    for scheme, n_act in (("scheme3", 5), ("scheme1", 8)):
        c = dict(cfg, action_scheme=scheme)
        whole = _make(1000, c, seed=77)
        part = _make(300, c, seed=77, env_offset=700)
        lib = whole.lib
        for step in (0, 1, 12345):
            a = whole.random_actions(step).cpu().numpy()
            b = part.random_actions(step).cpu().numpy()
            assert np.array_equal(a[700:], b)
            assert a.max() == n_act - 1 and a.min() == 0
            for e in (0, 1, 499, 999):
                for i in range(2):
                    u = lib.cz_spawn_uniform(77 ^ 0xA5A5A5A5A5A5A5A5, e, 0, step, i)
                    assert a[e, i] == int(u * n_act)
        counts = np.bincount(whole.random_actions(5).cpu().numpy().ravel(), minlength=n_act)
        assert counts.min() > 0.6 * 2000 / n_act
    # the stream drives a whole rollout without the host: 200 steps, every environment keeps stepping
    env = _make(4096, cfg, auto_reset=True, seed=3)
    env.reset()
    for t in range(200):
        env.step(env.random_actions(t))
    assert int(env.error_flags.abs().sum()) == 0 and int(env.info()["t"].max()) <= 50


@pytest.mark.parametrize("n", [333, 40011])
def test_host_buffer_step_matches_the_device_step(n):
    """cz_step_host (the reference-facing call with HOST buffers): small batches take one launch, batches of at least 32768
    environments are stepped as four column ranges whose device->host copies overlap the next range's kernels"""
    import ctypes as C
    from cooking_zoo_b200 import _native
    cfg = dict(level="coop_test", meta_file="example", num_agents=2, max_steps=20,
               recipes=["TomatoLettuceSalad", "CarrotBanana"], end_all=True, reward_scheme=None)
    a = _make(n, cfg, auto_reset=True, seed=6, layout_pool_size=64)
    b = _make(n, cfg, auto_reset=True, seed=6, layout_pool_size=64)
    a.reset(); b.reset()
    L = a.obs_len
    h_obs = torch.empty((n, 2, L), dtype=torch.float64).pin_memory()
    h_rew = torch.empty((n, 2), dtype=torch.float64).pin_memory()
    h_te = torch.empty((n, 2), dtype=torch.uint8).pin_memory()
    h_tr = torch.empty((n, 2), dtype=torch.uint8).pin_memory()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator().manual_seed(n)
    for t in range(25):
        act = torch.randint(0, 5, (n, 2), generator=g, dtype=torch.uint8).pin_memory()
        _native.check(b.lib.cz_step_host(b._handle, b.state.data_ptr(), act.data_ptr(), h_obs.data_ptr(), h_rew.data_ptr(),
                                         h_te.data_ptr(), h_tr.data_ptr(), n, _native.STEP_AUTO_RESET, 6, 0, stream))
        oa, ra, ta, ua, _ = a.step(act)
        assert torch.equal(oa.cpu().view(torch.int64), h_obs.view(torch.int64)), t
        assert torch.equal(ra.cpu().view(torch.int64), h_rew.view(torch.int64)), t
        assert torch.equal(ta.cpu(), h_te) and torch.equal(ua.cpu(), h_tr), t
    assert torch.equal(a.state, b.state)


def test_generic_tables_large_batch_any_plan_writer(monkeypatch, tmp_path):
    """tables outside the packed class step large batches as the generic dynamics kernel + cz_obs_any_kernel (warp per
    environment, any observation plan); CZ_ANY_WRITER=0 keeps the fused generic kernel.  Checked on the headline tables
    forced generic (against the specialised kernels) and on random / rich levels whose plans are really outside the class
    (more than 64 pairs, long table runs, odd row lengths)."""
    import random
    from cooking_zoo_b200 import BatchedCookingEnv
    from tests.kitchens import _random_level, _random_meta, _rich_level
    cfg = dict(level="coop_test", meta_file="example", num_agents=2, max_steps=30,
               recipes=["TomatoLettuceSalad", "CarrotBanana"], end_all=True, reward_scheme=None)
    n = 50001
    a = _make(n, cfg, auto_reset=True, seed=8, layout_pool_size=64)
    monkeypatch.setenv("CZ_GENERIC", "1")
    b = _make(n, cfg, auto_reset=True, seed=8, layout_pool_size=64)
    monkeypatch.delenv("CZ_GENERIC")
    a.reset(); b.reset()
    rng = np.random.default_rng(2)
    for t in range(35):
        act = torch.from_numpy(rng.integers(0, 5, size=(n, 2)).astype(np.uint8)).cuda()
        oa, ra, ta, ua, _ = a.step(act)
        l0 = b.lib.cz_launch_count()
        ob, rb, tb, ub, _ = b.step(act)
        assert b.lib.cz_launch_count() - l0 == 2
        assert torch.equal(oa.view(torch.int64), ob.view(torch.int64)), t
        assert torch.equal(ra.view(torch.int64), rb.view(torch.int64)) and torch.equal(ta, tb) and torch.equal(ua, ub)
    assert torch.equal(a.state, b.state)
    a.close(); b.close()
    seen_odd = seen_many_pairs = False
    for seed in (5003, 5005, 5006, 5020, 6001, 6004):
        r = random.Random(seed)
        lp, mp = str(tmp_path / f"level_{seed}.json"), str(tmp_path / f"meta_{seed}.json")
        if seed >= 6000:
            level = _random_level(r, lp)
            _random_meta(r, level, mp)
            A = 4
        else:
            _rich_level(r, lp, mp)
            A = r.randint(1, 2)
        recipes = ["TomatoLettuceSalad", "CarrotBanana", "TomatoSalad", "no_recipe"][:A]

        def make():
            e = BatchedCookingEnv(49152 + 77, lp, mp, A, 20, recipes, end_condition_all_dishes=True, action_scheme="scheme3",
                                  layout_pool_size=32, layout_seed=seed, auto_reset=True, seed=seed)
            e.reset()
            return e
        x = make()
        tb_ = x.tables
        packed = (tb_.num_agents * tb_.num_comp_slots <= 64 and tb_.num_obs_ranges == 1 and tb_.obs_table_len <= 128
                  and tb_.obs_len % 2 == 0)
        if packed:
            x.close()
            continue
        seen_odd |= tb_.obs_len % 2 == 1
        seen_many_pairs |= tb_.num_agents * tb_.num_comp_slots > 64
        monkeypatch.setenv("CZ_ANY_WRITER", "0")
        y = make()
        monkeypatch.delenv("CZ_ANY_WRITER")
        for t in range(25):
            act = torch.from_numpy(rng.integers(0, 5, size=(x.num_envs, A)).astype(np.uint8)).cuda()
            ox, rx, tx, ux, _ = x.step(act)
            oy, ry, ty, uy, _ = y.step(act)
            assert torch.equal(ox.view(torch.int64), oy.view(torch.int64)), (seed, t)
            assert torch.equal(rx.view(torch.int64), ry.view(torch.int64)) and torch.equal(tx, ty) and torch.equal(ux, uy)
        assert torch.equal(x.state, y.state)
        x.close(); y.close()
    assert seen_odd and seen_many_pairs
