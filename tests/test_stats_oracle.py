"""CPU: the episode-statistics rule of CZ_STEP_EPISODE_STATS (oracle/cz_stats.py) on hand-built step sequences, and driven
by the Python oracle on a random kitchen.  tests/test_gpu_episode_stats.py holds the device to the same function."""
import numpy as np

from oracle import cz_stats
from oracle.cz_oracle import OracleEnv
from tests.kitchens import kitchen, kitchen_config


def _trace(steps, A=2, R=2):
    """steps: (episode, t, done, roots, rewards) per step of ONE environment -> the arrays of episode_stats_from_trace"""
    ep = np.array([[s[0]] for s in steps], np.uint32)
    t = np.array([[s[1]] for s in steps])
    done = np.array([[s[2]] for s in steps], bool)
    roots = np.array([[list(s[3]) + [0] * (R - len(s[3]))] for s in steps], bool)
    rew = np.array([[list(s[4]) if len(s) > 4 else [0.0] * A] for s in steps], np.float64)
    return rew, ep, t, done, roots


def test_auto_reset_step_is_not_counted_and_the_length_is_t():
    # episode 1: three steps, done on the third by time-up; then the auto-reset step (EPISODE + 1, t = 0, reward 0)
    rew, ep, t, done, roots = _trace([(1, 1, 0, (), (0.25, -1.0)), (1, 2, 0, (), (0.5, 2.0)), (1, 3, 1, (), (0.125, 4.0)),
                                      (2, 0, 0, (), (0.0, 0.0)), (2, 1, 0, (), (1.0, 1.0))])
    rec = cz_stats.episode_stats_from_trace(rew, ep, t, done, roots, end_all=False)
    assert rec["finished"].tolist() == [1]
    assert rec["last_len"].tolist() == [3]
    assert rec["last_ret"].tolist() == [[0.25 + 0.5 + 0.125, -1.0 + 2.0 + 4.0]]
    assert rec["ret"].tolist() == [[1.0, 1.0]]          # the new episode: the reset step added nothing
    assert rec["open"].tolist() == [1] and rec["episode"].tolist() == [2]
    assert rec["last_success"].tolist() == [0] and rec["last_served"].tolist() == [0]
    assert rec["totals"].tolist() == [1, 3, 0, 0, 0.875, 5.0]


def test_stepping_past_done_without_auto_reset_latches_once():
    steps = [(1, 1, 0, ()), (1, 2, 1, (1,), (20.0, 0.0))] + [(1, 2 + k, 1, (1,), (-1.0, -1.0)) for k in range(1, 6)]
    rec = cz_stats.episode_stats_from_trace(*_trace(steps), end_all=False)
    assert rec["finished"].tolist() == [1]
    assert rec["last_len"].tolist() == [2]
    assert rec["last_ret"].tolist() == [[20.0, 0.0]]
    assert rec["ret"].tolist() == [[20.0, 0.0]] and rec["open"].tolist() == [0]
    assert rec["totals"].tolist() == [1, 2, 1, 1, 20.0, 0.0]


def test_a_host_reset_mid_episode_drops_the_partial_episode():
    steps = [(1, 1, 0, (), (5.0, 5.0)), (1, 2, 0, (), (5.0, 5.0)),          # reset after two steps (EPISODE 1 -> 2)
             (2, 1, 0, (), (1.0, 2.0)), (2, 2, 1, (1, 1), (3.0, 4.0))]
    rec = cz_stats.episode_stats_from_trace(*_trace(steps), end_all=True)
    assert rec["finished"].tolist() == [1]
    assert rec["last_ret"].tolist() == [[4.0, 6.0]] and rec["last_len"].tolist() == [2]
    assert rec["last_served"].tolist() == [2] and rec["last_success"].tolist() == [1]


def test_clear_counts_an_unstarted_episode_and_not_a_running_one():
    base = cz_stats.new_record(2, 2)
    base["totals"][:] = 7.0
    base["finished"][:] = 3
    rec = cz_stats.clear(base, episode=[4, 9], t=[0, 5])
    assert rec["open"].tolist() == [1, 0] and rec["episode"].tolist() == [4, 9]
    assert rec["totals"].tolist() == [0.0] * 6 and rec["finished"].tolist() == [0, 0]
    # both environments finish their current episode on the next step, then start (and finish) one more
    rew = np.ones((3, 2, 2))
    rew[1] = 0.0                                                    # the auto-reset step
    ep = np.array([[4, 9], [5, 10], [5, 10]])
    t = np.array([[1, 6], [0, 0], [1, 1]])
    done = np.array([[1, 1], [0, 0], [1, 1]], bool)
    roots = np.zeros((3, 2, 1), bool)
    out = cz_stats.episode_stats_from_trace(rew, ep, t, done, roots, end_all=False, record=rec)
    assert out["finished"].tolist() == [2, 1]                       # env 1's running episode was not counted
    assert out["totals"].tolist() == [3, 1 + 1 + 1, 0, 0, 3.0, 3.0]
    assert rec["finished"].tolist() == [0, 0]                       # the record passed in is not modified


def test_success_against_time_up_for_both_end_conditions():
    cases = [  # end_all, roots at done, served, success
        (True, (1, 0), 1, 0), (True, (1, 1), 2, 1), (True, (0, 0), 0, 0),
        (False, (1, 0), 1, 1), (False, (0, 1), 1, 1), (False, (0, 0), 0, 0)]
    for end_all, roots, served, success in cases:
        rec = cz_stats.episode_stats_from_trace(*_trace([(1, 1, 0, ()), (1, 2, 1, roots)]), end_all=end_all)
        assert rec["last_served"].tolist() == [served] and rec["last_success"].tolist() == [success], (end_all, roots)
        assert rec["totals"][2:4].tolist() == [served, success]


def test_served_counts_only_the_recipes_of_the_environment():
    marks = np.array([0x01010101, 0x00000001, 0x00020100, 0x010202FE], np.uint64)
    t, done, roots = cz_stats.decode_misc(np.full(4, 7 | 1 << 20), marks, 3)
    assert t.tolist() == [7] * 4 and done.all()
    assert roots.sum(-1).tolist() == [3, 1, 1, 0]     # byte 3 belongs to no recipe when R = 3; only bit 0 is the root


def test_totals_are_the_sums_of_the_latched_values():
    rng = np.random.default_rng(0)
    K, N, A, R = 60, 50, 3, 2
    rew = rng.normal(size=(K, N, A))
    ep = np.zeros((K, N), np.int64)
    t = np.zeros((K, N), np.int64)
    done = np.zeros((K, N), bool)
    e, c = np.ones(N, np.int64), np.zeros(N, np.int64)
    for k in range(K):
        reset = rng.random(N) < 0.1
        e, c = np.where(reset, e + 1, e), np.where(reset, 0, c + 1)
        ep[k], t[k] = e, c
        done[k] = (c >= 4) & (rng.random(N) < 0.5)
    roots = rng.random((K, N, R)) < 0.4
    rec = cz_stats.new_record(N, A)
    want = np.zeros(4 + A)
    for k in range(K):                      # step by step, summing whatever gets latched
        before = rec["finished"].copy()
        rec = cz_stats.episode_stats_from_trace(rew[k:k + 1], ep[k:k + 1], t[k:k + 1], done[k:k + 1], roots[k:k + 1],
                                                end_all=True, record=rec)
        f = rec["finished"] != before
        want += np.concatenate([[f.sum(), rec["last_len"][f].sum(), rec["last_served"][f].sum(),
                                 rec["last_success"][f].sum()], rec["last_ret"][f].sum(0)])
    whole = cz_stats.episode_stats_from_trace(rew, ep, t, done, roots, end_all=True)
    assert whole["finished"].sum() > 20
    assert np.array_equal(whole["totals"][:4], want[:4])
    np.testing.assert_allclose(whole["totals"][4:], want[4:], rtol=1e-12)
    for k in ("ret", "last_ret", "last_len", "last_served", "last_success", "finished", "episode", "open"):
        assert np.array_equal(whole[k], rec[k]), k


def test_the_python_oracle_on_a_random_kitchen_with_resets(tmp_path):
    from cooking_zoo_b200.tables import compile_tables
    seed, max_steps, steps = 3, 5, 80
    lp, mp, _ = kitchen(seed, str(tmp_path))
    cfg = kitchen_config(seed)
    cfg["spawn"] = None
    A = cfg["A"]
    t_ = compile_tables(lp, mp, A, max_steps, cfg["recipes"], layout_pool_size=2, layout_seed=seed)
    env = OracleEnv(t_.layouts[0], cfg["recipes"], max_steps, end_condition_all_dishes=cfg["end_all"],
                    action_scheme=cfg["scheme"])
    n_act = 8 if cfg["scheme"] == "scheme1" else 5
    rng = np.random.default_rng(seed)
    episode, resets, lengths = 1, 0, []
    rec = cz_stats.clear(cz_stats.new_record(1, A), [episode], [0])
    for _ in range(steps):
        if env.t >= max_steps or any(env.terminated):   # the caller resets a finished environment: EPISODE + 1
            env.reset()
            episode += 1
            resets += 1
        r, te, _, _ = env.step(rng.integers(0, n_act, size=A))
        comp = [rec_[0].marked for rec_ in env.recipes]
        done = env.t >= max_steps or (all(comp) if cfg["end_all"] else any(comp))
        if done:
            lengths.append(env.t)
        rec = cz_stats.episode_stats_from_trace(np.array([[r]], np.float64), [[episode]], [[env.t]], [[done]], [[comp]],
                                                cfg["end_all"], record=rec)
        if done:
            assert rec["last_len"].tolist() == [env.t]
    assert resets >= steps // max_steps - 1
    assert rec["finished"].tolist() == [len(lengths)]
    assert rec["finished"][0] in (resets, resets + 1)                 # every reset followed a finished episode
    assert rec["totals"][0] == len(lengths) and rec["totals"][1] == sum(lengths)
