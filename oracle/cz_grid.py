"""Grid observation from the canonical state arrays: the checker of cz_observe_grid (include/cz_b200.h).

TEST INFRASTRUCTURE ONLY, like the rest of oracle/: it does not import cooking_zoo_b200.  It reads the canonical arrays that
the golden traces store and that OracleEnv.export_state, CEnv.export_state and BatchedCookingEnv.export_state return
(oracle/ref_dump.py documents them), so one function serves reference-recorded states and both oracles.

Channel order for observer a (restated from cz_b200.h): 7 static kinds (floor, counter, cutboard, blender, deliversquare,
switch, block), 5 static states (cutboard_ready, blender_ready, blender_on, switch_active, block_walkable), n:<Type> for every
dynamic type of the meta file in meta order, chopped:<Type> / mashed:<Type> for the choppable / blendable ones, on_plate, then
one group of 7 planes per agent: group 0 is agent a, then the other agents in ascending index.
"""
import numpy as np

from .cz_oracle import TRAITS

STATIC_KINDS = ("Floor", "Counter", "Cutboard", "Blender", "Deliversquare", "Switch", "Block")
STATE_CHANNELS = ("cutboard_ready", "blender_ready", "blender_on", "switch_active", "block_walkable")


def _dyn_types(meta):
    return [name for name, _ in meta if TRAITS[name]["kind"] == "dynamic"]


def grid_channel_names(meta, A):
    """Channel names for a meta file ([(type name, count)], meta order) and A agents."""
    types = _dyn_types(meta)
    names = [k.lower() for k in STATIC_KINDS] + list(STATE_CHANNELS)
    names += [f"n:{n}" for n in types]
    names += [f"chopped:{n}" for n in types if TRAITS[n].get("chop")]
    names += [f"mashed:{n}" for n in types if TRAITS[n].get("blend")]
    names.append("on_plate")
    for g in range(A):
        names += [f"agent{g}"] + [f"agent{g}_facing{o}" for o in range(1, 5)] + [f"agent{g}_holding", f"agent{g}_active"]
    return names


def grid_from_state(state, meta, A, W, H):
    """uint8 [A, C, H, W] grid of every observer from the canonical arrays `agents` [A, 6], `objs` [D, 9], `statics` [S, 4].

    Static kinds and positions come from the `statics` rows (the slot's type from the meta order); floor is every cell of
    the W x H grid that no other static occupies."""
    return grid_from_states([state], meta, A, W, H)[0]


def grid_from_states(states, meta, A, W, H):
    """grid_from_state of a list of states of the same tables -> uint8 [n, A, C, H, W] (vectorised over the states)."""
    names = grid_channel_names(meta, A)
    ch = {nm: i for i, nm in enumerate(names)}
    C, n = len(names), len(states)
    agents = np.stack([np.asarray(s["agents"], np.int64) for s in states]).reshape(n, A, 6)
    statics = np.stack([np.asarray(s["statics"], np.int64) for s in states]).reshape(n, -1, 4)
    objs = np.stack([np.asarray(s["objs"], np.int64) for s in states]).reshape(n, -1, 9)
    shared = np.zeros((n, C, H, W), np.int64)       # the observer-independent planes
    env = np.arange(n)[:, None]
    # statics: slot type from the meta order; Floor slots are left to the floor rule
    slot_kind = [name for name, num in meta if TRAITS[name]["kind"] == "static" for _ in range(num)]
    if slot_kind:
        kind_ch = np.array([ch[k.lower()] if k != "Floor" else -1 for k in slot_kind])
        pres = (statics[:, :, 0] == 1) & (kind_ch >= 0)[None]
        x, y, bits = statics[:, :, 1], statics[:, :, 2], statics[:, :, 3]
        e = np.broadcast_to(env, pres.shape)
        kc = np.broadcast_to(kind_ch[None], pres.shape)
        np.add.at(shared, (e[pres], kc[pres], y[pres], x[pres]), 1)
        for kind, bit, name in (("Cutboard", 1, "cutboard_ready"), ("Blender", 1, "blender_ready"), ("Blender", 2, "blender_on"),
                                ("Switch", 4, "switch_active"), ("Block", 8, "block_walkable")):
            m = pres & (np.array([k == kind for k in slot_kind])[None]) & ((bits & bit) != 0)
            shared[e[m], ch[name], y[m], x[m]] = 1
    shared[:, ch["floor"]] = shared[:, :7].sum(1) == 0
    # dynamic objects: slot type from the meta order
    slot_type = [name for name, num in meta if TRAITS[name]["kind"] == "dynamic" for _ in range(num)]
    if slot_type:
        def chan(prefix, trait=None):
            return np.array([ch[f"{prefix}:{t}"] if trait is None or TRAITS[t].get(trait) else -1 for t in slot_type])
        pres = objs[:, :, 0] == 1
        x, y = objs[:, :, 1], objs[:, :, 2]
        e = np.broadcast_to(env, pres.shape)
        for c_of_slot, cond in ((chan("n"), pres), (chan("chopped", "chop"), pres & (objs[:, :, 3] != 0)),
                                (chan("mashed", "blend"), pres & (objs[:, :, 4] == 2))):
            cs = np.broadcast_to(c_of_slot[None], pres.shape)
            m = cond & (cs >= 0)
            np.add.at(shared, (e[m], cs[m], y[m], x[m]), 1)
        m = pres & (objs[:, :, 6] == 2)
        np.add.at(shared, (e[m], ch["on_plate"], y[m], x[m]), 1)
    out = np.repeat(shared[:, None].astype(np.uint8), A, axis=1)
    g0 = ch["agent0"]
    for a in range(A):
        for g, i in enumerate([a] + [j for j in range(A) if j != a]):
            x, y, o, holding, active = (agents[:, i, k] for k in range(5))
            on = (x >= 0) & (x < W) & (y >= 0) & (y < H)
            e, xs, ys = np.nonzero(on)[0], x[on], y[on]
            base = g0 + 7 * g
            out[e, a, base, ys, xs] = 1
            f = (o[on] >= 1) & (o[on] <= 4)
            out[e[f], a, base + o[on][f], ys[f], xs[f]] = 1
            f = holding[on] >= 0
            out[e[f], a, base + 5, ys[f], xs[f]] = 1
            f = active[on] != 0
            out[e[f], a, base + 6, ys[f], xs[f]] = 1
    return out
