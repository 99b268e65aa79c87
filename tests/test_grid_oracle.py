"""CPU: the grid observation's oracle (oracle/cz_grid.py) against the library's channel names, the golden traces and a
directed kitchen whose grids are stated element by element."""
import json

import numpy as np
import pytest

from oracle.cz_grid import grid_channel_names, grid_from_state
from oracle.cz_oracle import OracleEnv, TRAITS
from tests.kitchens import DEVICE_KITCHENS, kitchen
from tests.replay import golden_files, load_golden


def _meta_pairs(path):
    return [next(iter(e.items())) for e in json.load(open(path))]


def test_channel_names_match_the_library_for_the_shipped_meta():
    from cooking_zoo_b200.grid import grid_channels
    from cooking_zoo_b200.levels import load_meta
    from cooking_zoo_b200.tables import compile_tables
    for A in (1, 2):
        t = compile_tables("coop_test", "example", A, 100, ["TomatoSalad"] * A, layout_pool_size=2)
        names = grid_channels(t)
        assert names == grid_channel_names(load_meta("example"), A)
        assert len(names) == 7 + 5 + 9 + 8 + 2 + 1 + 7 * A          # 46 for two agents
    assert grid_channel_names(load_meta("example"), 2)[12:21] == [
        "n:Plate", "n:Tomato", "n:Onion", "n:Lettuce", "n:Carrot", "n:Banana", "n:Apple", "n:Watermelon", "n:Bread"]


@pytest.mark.parametrize("seed", DEVICE_KITCHENS[::3])
def test_channel_names_match_the_library_on_random_kitchens(seed, tmp_path):
    from cooking_zoo_b200.grid import grid_channels
    from cooking_zoo_b200.tables import compile_tables
    lp, mp, level = kitchen(seed, str(tmp_path))
    max_agents = sum(e.get("MAX_COUNT", 1) for e in level["AGENTS"])
    for A in range(1, min(4, max_agents) + 1):
        t = compile_tables(lp, mp, A, 50, ["TomatoSalad"] * A, layout_pool_size=2, layout_seed=seed)
        assert grid_channels(t) == grid_channel_names(_meta_pairs(mp), A), (seed, A)


def _golden_states():
    for path in golden_files():
        g = load_golden(path)
        A = g["config"]["num_agents"]
        for n, layout in enumerate(g["layouts"]):
            for t in range(int(g["length"][n]) + 1):
                yield path, n, t, layout, A, {k: g[k][n, t] for k in ("agents", "objs", "statics")}


def test_golden_states_give_consistent_grids():
    """On every state of every golden trace: one static kind per cell, the object counts, the agent planes, and group 0
    of observer a is agent a."""
    count = 0
    for path, n, t, layout, A, st in _golden_states():
        ctx = f"{path} trace {n} state {t}"
        meta, W, H = layout["meta"], layout["width"], layout["height"]
        names = grid_channel_names(meta, A)
        grid = grid_from_state(st, meta, A, W, H)
        assert grid.shape == (A, len(names), H, W), ctx
        assert (grid[:, :7].sum(1) == 1).all(), ctx
        slot_type = [name for name, num in meta if TRAITS[name]["kind"] == "dynamic" for _ in range(num)]
        objs = st["objs"]
        for typ in set(slot_type):
            want = sum(1 for s, ty in enumerate(slot_type) if ty == typ and objs[s, 0])
            assert (grid[:, names.index(f"n:{typ}")].sum((1, 2)) == want).all(), (ctx, typ)
        assert (grid[:, names.index("on_plate")].sum((1, 2)) == int(((objs[:, 0] == 1) & (objs[:, 6] == 2)).sum())).all(), ctx
        g0 = names.index("agent0")
        for a in range(A):
            order = [a] + [i for i in range(A) if i != a]
            for g, i in enumerate(order):
                x, y, o, holding, active, _ = st["agents"][i].tolist()
                planes = grid[a, g0 + 7 * g:g0 + 7 * g + 7]
                want = np.zeros((7, H, W), np.uint8)
                want[0, y, x] = 1
                if 1 <= o <= 4:
                    want[o, y, x] = 1
                want[5, y, x] = holding >= 0
                want[6, y, x] = active
                assert np.array_equal(planes, want), (ctx, a, g)
        count += 1
    assert count > 1000


# a directed kitchen: C counter, D deliversquare, K cutboard, B blender, S switch, X block, . floor
MAP = ["CCDCC",
       "K...C",
       "C.S.B",
       "C...C",
       "CXCCC"]
KIND = {"C": "Counter", "D": "Deliversquare", "K": "Cutboard", "B": "Blender", "S": "Switch", "X": "Block", ".": "Floor"}
META = [["Cutboard", 1], ["Counter", 20], ["Blender", 1], ["Deliversquare", 1], ["Plate", 1], ["Tomato", 1], ["Onion", 1],
        ["Carrot", 1], ["Agent", 2], ["Block", 1], ["Switch", 1]]
# (event, actions of agents 0 and 1, every non-zero element of observer 0's grid outside the 7 static kind planes after the
# step: "channel@x,y" is 1, "channel@x,y=n" is n).  Actions (scheme3): 1 left, 2 right, 3 down, 4 up; walking into a
# non-walkable cell interacts with it.
SCRIPT = [
    ("reset", None,
     "n:Plate@4,1 n:Tomato@0,2 n:Carrot@4,3 agent0@1,2 agent0_facing1@1,2 agent0_active@1,2 agent1@3,2 agent1_facing1@3,2 "
     "agent1_active@3,2"),
    ("pick-up", [1, 0],
     "n:Plate@4,1 n:Tomato@1,2 n:Carrot@4,3 agent0@1,2 agent0_facing1@1,2 agent0_holding@1,2 agent0_active@1,2 agent1@3,2 "
     "agent1_facing1@3,2 agent1_active@3,2"),
    ("walk up", [4, 0],
     "n:Plate@4,1 n:Tomato@1,1 n:Carrot@4,3 agent0@1,1 agent0_facing4@1,1 agent0_holding@1,1 agent0_active@1,1 agent1@3,2 "
     "agent1_facing1@3,2 agent1_active@3,2"),
    ("put on the cutboard", [1, 0],
     "cutboard_ready@0,1 n:Plate@4,1 n:Tomato@0,1 n:Carrot@4,3 agent0@1,1 agent0_facing1@1,1 agent0_active@1,1 agent1@3,2 "
     "agent1_facing1@3,2 agent1_active@3,2"),
    ("chop", [1, 0],
     "n:Plate@4,1 n:Tomato@0,1 n:Carrot@4,3 chopped:Tomato@0,1 agent0@1,1 agent0_facing1@1,1 agent0_active@1,1 agent1@3,2 "
     "agent1_facing1@3,2 agent1_active@3,2"),
    ("pick up the chopped tomato", [1, 0],
     "n:Plate@4,1 n:Tomato@1,1 n:Carrot@4,3 chopped:Tomato@1,1 agent0@1,1 agent0_facing1@1,1 agent0_holding@1,1 "
     "agent0_active@1,1 agent1@3,2 agent1_facing1@3,2 agent1_active@3,2"),
    ("walk right / down", [2, 3],
     "n:Plate@4,1 n:Tomato@2,1 n:Carrot@4,3 chopped:Tomato@2,1 agent0@2,1 agent0_facing2@2,1 agent0_holding@2,1 "
     "agent0_active@2,1 agent1@3,3 agent1_facing3@3,3 agent1_active@3,3"),
    ("walk right", [2, 0],
     "n:Plate@4,1 n:Tomato@3,1 n:Carrot@4,3 chopped:Tomato@3,1 agent0@3,1 agent0_facing2@3,1 agent0_holding@3,1 "
     "agent0_active@3,1 agent1@3,3 agent1_facing3@3,3 agent1_active@3,3"),
    ("plate merge", [2, 0],
     "n:Plate@4,1 n:Tomato@4,1 n:Carrot@4,3 chopped:Tomato@4,1 on_plate@4,1 agent0@3,1 agent0_facing2@3,1 agent0_active@3,1 "
     "agent1@3,3 agent1_facing3@3,3 agent1_active@3,3"),
    ("agent 1 picks up the carrot", [0, 2],
     "n:Plate@4,1 n:Tomato@4,1 n:Carrot@3,3 chopped:Tomato@4,1 on_plate@4,1 agent0@3,1 agent0_facing2@3,1 agent0_active@3,1 "
     "agent1@3,3 agent1_facing2@3,3 agent1_holding@3,3 agent1_active@3,3"),
    ("agent 1 walks up", [0, 4],
     "n:Plate@4,1 n:Tomato@4,1 n:Carrot@3,2 chopped:Tomato@4,1 on_plate@4,1 agent0@3,1 agent0_facing2@3,1 agent0_active@3,1 "
     "agent1@3,2 agent1_facing4@3,2 agent1_holding@3,2 agent1_active@3,2"),
    ("put in the blender", [0, 2],
     "blender_ready@4,2 n:Plate@4,1 n:Tomato@4,1 n:Carrot@4,2 chopped:Tomato@4,1 on_plate@4,1 agent0@3,1 agent0_facing2@3,1 "
     "agent0_active@3,1 agent1@3,2 agent1_facing2@3,2 agent1_active@3,2"),
    # the toggle switches the blender on, which mashes the carrot in the same step and switches itself off
    ("blender toggle", [0, 2],
     "n:Plate@4,1 n:Tomato@4,1 n:Carrot@4,2 chopped:Tomato@4,1 mashed:Carrot@4,2 on_plate@4,1 agent0@3,1 agent0_facing2@3,1 "
     "agent0_active@3,1 agent1@3,2 agent1_facing2@3,2 agent1_active@3,2"),
    ("walk left", [1, 0],
     "n:Plate@4,1 n:Tomato@4,1 n:Carrot@4,2 chopped:Tomato@4,1 mashed:Carrot@4,2 on_plate@4,1 agent0@2,1 agent0_facing1@2,1 "
     "agent0_active@2,1 agent1@3,2 agent1_facing2@3,2 agent1_active@3,2"),
    ("switch press", [3, 0],
     "switch_active@2,2 block_walkable@1,4 n:Plate@4,1 n:Tomato@4,1 n:Carrot@4,2 chopped:Tomato@4,1 mashed:Carrot@4,2 "
     "on_plate@4,1 agent0@2,2 agent0_facing3@2,2 agent0_active@2,2 agent1@3,2 agent1_facing2@3,2 agent1_active@3,2"),
]


def _directed_layout():
    objs = {}
    for y, row in enumerate(MAP):
        for x, c in enumerate(row):
            objs.setdefault(KIND[c], []).append([x, y])
    dyn = [["Plate", [[4, 1]]], ["Tomato", [[0, 2]]], ["Carrot", [[4, 3]]]]
    return {"width": 5, "height": 5, "meta": META, "objects": [[k, v] for k, v in objs.items()] + dyn,
            "agents": [[1, 2], [3, 2]]}


def _expected(text, names):
    want = np.zeros((len(names), 5, 5), np.uint8)
    for y, row in enumerate(MAP):
        for x, c in enumerate(row):
            want[names.index(KIND[c].lower()), y, x] = 1
    for item in text.split():
        ch, at = item.split("@")
        xy, _, v = at.partition("=")
        x, y = map(int, xy.split(","))
        want[names.index(ch), y, x] = int(v or 1)
    return want


def test_directed_kitchen_grids():
    env = OracleEnv(_directed_layout(), ["TomatoSalad", "CarrotBanana"], 100)
    names = grid_channel_names(META, 2)
    assert len(names) == 7 + 5 + 4 + 3 + 1 + 1 + 14
    for event, actions, text in SCRIPT:
        if actions is not None:
            env.step(actions)
        grid = grid_from_state(env.export_state(), META, 2, 5, 5)
        assert np.array_equal(grid[0], _expected(text, names)), event
        # observer 1 sees the same world with the agent groups swapped
        swapped = grid[0].copy()
        g0 = names.index("agent0")
        swapped[g0:g0 + 7], swapped[g0 + 7:g0 + 14] = grid[0, g0 + 7:g0 + 14], grid[0, g0:g0 + 7]
        assert np.array_equal(grid[1], swapped), event
    assert env.error == 0


def test_hand_made_state_counts_and_blender_on():
    """counts above one, a blender that is on, and an inactive agent, from canonical arrays written by hand"""
    names = grid_channel_names(META, 2)
    statics = OracleEnv(_directed_layout(), ["TomatoSalad"], 100).export_state()["statics"]
    assert statics[21].tolist() == [1, 4, 2, 0]
    statics[21] = (1, 4, 2, 3)                     # Blender: ready and on
    objs = np.zeros((4, 9), np.int16)
    objs[0] = (1, 3, 3, 0, 0, 0, 0, 1, 0)          # Plate held by agent 1
    objs[1] = (1, 3, 3, 1, 0, 1, 2, 0, 0)          # chopped Tomato on that plate
    objs[2] = (1, 3, 3, 0, 0, 1, 2, 0, 1)          # Onion on that plate
    objs[3] = (1, 4, 2, 0, 2, 1, 1, 14, 0)         # mashed Carrot in the blender
    agents = np.array([[1, 1, 3, -1, 0, 5], [3, 3, 2, 0, 1, 0]], np.int16)
    grid = grid_from_state({"agents": agents, "objs": objs, "statics": statics}, META, 2, 5, 5)
    want = _expected("blender_ready@4,2 blender_on@4,2 n:Plate@3,3 n:Tomato@3,3 n:Onion@3,3 n:Carrot@4,2 chopped:Tomato@3,3 "
                     "mashed:Carrot@4,2 on_plate@3,3=2 agent0@1,1 agent0_facing3@1,1 agent1@3,3 agent1_facing2@3,3 "
                     "agent1_holding@3,3 agent1_active@3,3", names)
    assert np.array_equal(grid[0], want)
