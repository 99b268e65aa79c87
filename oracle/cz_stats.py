"""Episode statistics of CZ_STEP_EPISODE_STATS (include/cz_b200.h) over per-step arrays, in numpy.

Imports nothing from the package, so one function serves the golden traces, both oracles and the device tests.  The
rule, after every step of every environment, with the post-step EPISODE counter, clock t, done bit and recipe-root marks
and that step's rewards r[a]:
  1. EPISODE != record episode (a reset since the last step): episode = EPISODE, ret = 0, open = 1;
  2. open: ret += r (float64, in step order);
  3. open and done: last_ret = ret, last_len = t, last_served = roots set, last_success = all roots (end_all) or any
     root, finished += 1, totals += (1, t, served, success, ret), open = 0.
clear(): ret, the last_* fields, finished and the totals become 0, episode = EPISODE, open = (t == 0).
"""
import numpy as np

TI_DONE = 1 << 20
FIELDS = ("ret", "episode", "open", "last_ret", "last_len", "last_served", "last_success", "finished", "totals")


def new_record(n, num_agents):
    """an all-zero record for n environments of num_agents agents"""
    return {"ret": np.zeros((n, num_agents), np.float64), "episode": np.zeros(n, np.uint32), "open": np.zeros(n, np.uint8),
            "last_ret": np.zeros((n, num_agents), np.float64), "last_len": np.zeros(n, np.int32),
            "last_served": np.zeros(n, np.uint8), "last_success": np.zeros(n, np.uint8), "finished": np.zeros(n, np.int32),
            "totals": np.zeros(4 + num_agents, np.float64)}


def clear(record, episode, t):
    """the clear rule on a record (modified in place and returned): episode [N] and t [N] of the current state"""
    for k in ("ret", "last_ret", "last_len", "last_served", "last_success", "finished", "totals"):
        record[k][...] = 0
    record["episode"][...] = np.asarray(episode, np.uint32)
    record["open"][...] = (np.asarray(t) == 0).astype(np.uint8)
    return record


def decode_misc(tinfo, marks, num_recipes):
    """(t, done, roots [..., R]) from TINFO and MARKS words"""
    tinfo = np.asarray(tinfo, np.uint64)
    marks = np.asarray(marks, np.uint64)
    t = (tinfo & 0xFFFFF).astype(np.int64)
    done = ((tinfo >> 20) & 1).astype(bool)
    roots = np.stack([((marks >> (8 * r)) & 1).astype(bool) for r in range(num_recipes)], -1)
    return t, done, roots


def episode_stats_from_trace(rewards, episode, t, done, roots, end_all, record=None):
    """The rule over K steps.  rewards f64 [K, N, A]; episode [K, N], t [K, N], done [K, N] and roots [K, N, R] (bool: root
    mark of recipe r) of the post-step states; end_all: end_condition_all_dishes.  record: the record before the first step
    (default: all zero), not modified.  Returns the record after the last step (every field, the totals included)."""
    rewards = np.asarray(rewards, np.float64)
    K, N, A = rewards.shape
    episode = np.asarray(episode).astype(np.uint32).reshape(K, N)
    t = np.asarray(t).astype(np.int64).reshape(K, N)
    done = np.asarray(done).astype(bool).reshape(K, N)
    roots = np.asarray(roots).astype(bool).reshape(K, N, -1)
    R = roots.shape[-1]
    rec = new_record(N, A) if record is None else {k: np.array(v, copy=True) for k, v in record.items()}
    for k in range(K):
        new = episode[k] != rec["episode"]
        rec["episode"][new] = episode[k][new]
        rec["ret"][new] = 0.0
        rec["open"][new] = 1
        op = rec["open"] != 0
        rec["ret"][op] = rec["ret"][op] + rewards[k][op]
        fin = op & done[k]
        if not fin.any():
            continue
        served = roots[k].sum(-1)
        success = (served == R) if end_all else (served > 0)
        rec["last_ret"][fin] = rec["ret"][fin]
        rec["last_len"][fin] = t[k][fin]
        rec["last_served"][fin] = served[fin]
        rec["last_success"][fin] = success[fin]
        rec["finished"][fin] += 1
        rec["open"][fin] = 0
        rec["totals"][0] += fin.sum()
        rec["totals"][1] += t[k][fin].sum()
        rec["totals"][2] += served[fin].sum()
        rec["totals"][3] += success[fin].sum()
        rec["totals"][4:] += rec["ret"][fin].sum(0)
    return rec
