"""Random kitchen generators shared by the tests (a helper module, not a test file).

_random_level / _random_meta: open kitchens up to 8x8 with random inner counters, appliances and ingredients on the
counter ring, OPTIONAL objects and a meta file with random counts in random order.  _rich_level: an 8x8 kitchen with
many objects and a meta file in the order of example.json; _lean_level: the same with few objects.  served_recipes: the book recipes a kitchen can serve."""
import json
import os
import random

from oracle.cz_oracle import RECIPES, make_recipe

BOOK = list(RECIPES)


def _random_level(rng, path, split=False):
    """an open kitchen: counter ring, random inner counters, appliances on the ring, ingredients on counters.
    split=True adds an inner counter wall (a full column of the floor) that cuts the floor in two: agents on one side
    reach only the ring cells of their side, which is what the cook's reachability tables and its "nothing reachable"
    crashes are about."""
    W, H = rng.randint(5, 8), rng.randint(5, 8)
    rows = [["-"] * W] + [["-"] + [" "] * (W - 2) + ["-"] for _ in range(H - 2)] + [["-"] * W]
    for _ in range(rng.randint(0, 3)):
        rows[rng.randint(2, H - 3)][rng.randint(2, W - 3)] = "-"
    if split:
        x = rng.randint(2, W - 3)
        for y in range(1, H - 1):
            rows[y][x] = "-"
    ring = [(x, 0) for x in range(1, W - 1)] + [(x, H - 1) for x in range(1, W - 1)] + \
           [(0, y) for y in range(1, H - 1)] + [(W - 1, y) for y in range(1, H - 1)]
    rng.shuffle(ring)
    statics = []
    for name, count in (("Cutboard", rng.randint(1, 2)), ("Blender", rng.randint(0, 1)), ("Deliversquare", rng.randint(1, 2))):
        for _ in range(count):
            x, y = ring.pop()
            statics.append({name: {"COUNT": 1, "X_POSITION": [x], "Y_POSITION": [y]}})
    foods = ["Plate", "Plate", "Tomato", "Lettuce", "Carrot", "Banana", "Bread", "Onion", "Apple", "Watermelon"]
    rng.shuffle(foods)
    dyn = []
    for name in foods[:rng.randint(3, 8)]:
        x, y = ring.pop()          # one cell per entry: a cross product of two ring cells could name a taken or a floor cell
        entry = {"COUNT": 1, "X_POSITION": [x], "Y_POSITION": [y]}
        if rng.random() < 0.2:
            entry["OPTIONAL"] = 0.5
        dyn.append({name: entry})
    agents = [{"MAX_COUNT": 2, "X_POSITION": list(range(1, W - 1)), "Y_POSITION": list(range(1, H - 1))},
              {"MAX_COUNT": 2, "X_POSITION": list(range(1, W - 1)), "Y_POSITION": list(range(1, H - 1))}]
    level = {"LEVEL_LAYOUT": "\n".join("".join(r) for r in rows), "STATIC_OBJECTS": statics, "DYNAMIC_OBJECTS": dyn,
             "AGENTS": agents, "DYNAMIC_EXCLUDED_POSITIONS": []}
    json.dump(level, open(path, "w"))
    return level


def _random_meta(rng, level, path):
    need = {}
    for group in ("STATIC_OBJECTS", "DYNAMIC_OBJECTS"):
        for entry in level[group]:
            (name, spec), = entry.items()
            need[name] = need.get(name, 0) + spec["COUNT"]
    order = ["Cutboard", "Counter", "Blender", "Deliversquare", "Plate", "Tomato", "Onion", "Lettuce", "Carrot", "Banana",
             "Apple", "Watermelon", "Bread", "Agent", "Block", "Switch"]
    rng.shuffle(order)
    meta = []
    for name in order:
        lo = need.get(name, 0) + (1 if name == "Bread" and need.get(name, 0) else 0)       # room for a chopped twin
        if name == "Counter":
            lo = 64
        if name == "Agent":
            lo = 4
        meta.append({name: lo + rng.randint(0, 2)})
    json.dump(meta, open(path, "w"))


def _rich_level(rng, lp, mp):
    """an 8x8 kitchen with many objects (more than 16 live dynamic slots: one environment per warp) and a meta file in
    the order of example.json (packed observation plan: the specialised kernels)"""
    W = H = 8
    rows = [["-"] * W] + [["-"] + [" "] * (W - 2) + ["-"] for _ in range(H - 2)] + [["-"] * W]
    ring = [(x, 0) for x in range(1, W - 1)] + [(x, H - 1) for x in range(1, W - 1)] + \
           [(0, y) for y in range(1, H - 1)] + [(W - 1, y) for y in range(1, H - 1)]
    rng.shuffle(ring)
    statics, need = [], {}
    for name, count in (("Cutboard", 2), ("Blender", 1), ("Deliversquare", 2)):
        for _ in range(count):
            x, y = ring.pop()
            statics.append({name: {"COUNT": 1, "X_POSITION": [x], "Y_POSITION": [y]}})
            need[name] = need.get(name, 0) + 1
    dyn = []
    for name in ["Plate", "Tomato", "Onion", "Lettuce", "Carrot", "Banana", "Apple", "Watermelon", "Bread"]:
        for _ in range(rng.randint(1, 3)):
            if not ring:
                break
            x, y = ring.pop()
            dyn.append({name: {"COUNT": 1, "X_POSITION": [x], "Y_POSITION": [y]}})
            need[name] = need.get(name, 0) + 1
    level = {"LEVEL_LAYOUT": "\n".join("".join(r) for r in rows), "STATIC_OBJECTS": statics, "DYNAMIC_OBJECTS": dyn,
             "AGENTS": [{"MAX_COUNT": 4, "X_POSITION": list(range(1, W - 1)), "Y_POSITION": list(range(1, H - 1))}],
             "DYNAMIC_EXCLUDED_POSITIONS": []}
    json.dump(level, open(lp, "w"))
    meta = []
    for name in ["Cutboard", "Counter", "Blender", "Deliversquare", "Plate", "Tomato", "Onion", "Lettuce", "Carrot", "Banana",
                 "Apple", "Watermelon", "Bread", "Agent", "Block", "Switch"]:
        n = need.get(name, 0) + rng.randint(0, 1) + (need.get(name, 0) if name == "Bread" else 0)
        n_counters = 2 * W + 2 * (H - 2) - sum(need.get(k, 0) for k in ("Cutboard", "Blender", "Deliversquare"))
        meta.append({name: n_counters + rng.randint(0, 1) if name == "Counter" else (4 if name == "Agent" else n)})
    json.dump(meta, open(mp, "w"))
    return level


def _lean_level(rng, lp, mp):
    """a 5x5 to 8x8 kitchen with few objects (one to six kinds of food, one of each) and a meta file in the order of
    example.json: packed observation plans with few computed slots, so that 2-4 agents still have at most 32 (observer,
    slot) pairs (the specialised multi-agent kernels) or 33-64 (the two-pairs-per-lane writers)"""
    W, H = rng.randint(5, 8), rng.randint(5, 8)
    rows = [["-"] * W] + [["-"] + [" "] * (W - 2) + ["-"] for _ in range(H - 2)] + [["-"] * W]
    ring = [(x, 0) for x in range(1, W - 1)] + [(x, H - 1) for x in range(1, W - 1)] + \
           [(0, y) for y in range(1, H - 1)] + [(W - 1, y) for y in range(1, H - 1)]
    rng.shuffle(ring)
    statics, need = [], {}
    for name, count in (("Cutboard", rng.randint(1, 2)), ("Blender", rng.randint(0, 1)), ("Deliversquare", 1)):
        for _ in range(count):
            x, y = ring.pop()
            statics.append({name: {"COUNT": 1, "X_POSITION": [x], "Y_POSITION": [y]}})
            need[name] = need.get(name, 0) + 1
    foods = ["Tomato", "Onion", "Lettuce", "Carrot", "Banana", "Apple", "Watermelon", "Bread"]
    dyn = []
    for name in ["Plate"] + rng.sample(foods, rng.randint(1, 6)):
        x, y = ring.pop()
        dyn.append({name: {"COUNT": 1, "X_POSITION": [x], "Y_POSITION": [y]}})
        need[name] = 1
    level = {"LEVEL_LAYOUT": "\n".join("".join(r) for r in rows), "STATIC_OBJECTS": statics, "DYNAMIC_OBJECTS": dyn,
             "AGENTS": [{"MAX_COUNT": 4, "X_POSITION": list(range(1, W - 1)), "Y_POSITION": list(range(1, H - 1))}],
             "DYNAMIC_EXCLUDED_POSITIONS": []}
    json.dump(level, open(lp, "w"))
    n_counters = 2 * W + 2 * (H - 2) - sum(need.get(k, 0) for k in ("Cutboard", "Blender", "Deliversquare"))
    meta = []
    for name in ["Cutboard", "Counter", "Blender", "Deliversquare", "Plate", "Tomato", "Onion", "Lettuce", "Carrot", "Banana",
                 "Apple", "Watermelon", "Bread", "Agent", "Block", "Switch"]:
        n = need.get(name, 0) + rng.randint(0, 1) + (need.get(name, 0) if name == "Bread" else 0)
        meta.append({name: n_counters + rng.randint(0, 1) if name == "Counter" else (4 if name == "Agent" else n)})
    json.dump(meta, open(mp, "w"))
    return level


def kitchen(seed, directory):
    """kitchen `seed` of the random-kitchen tests -> (level path, meta path, level dict): seeds from 1000 on a lean
    kitchen; below, seed % 4 == 0 a rich kitchen, 1 a random kitchen split in two by an inner wall, 2 and 3 a random
    open kitchen"""
    rng = random.Random(seed)
    lp, mp = os.path.join(directory, f"level_{seed}.json"), os.path.join(directory, f"meta_{seed}.json")
    if seed >= 1000:
        level = _lean_level(rng, lp, mp)
    elif seed % 4 == 0:
        level = _rich_level(rng, lp, mp)
    else:
        level = _random_level(rng, lp, split=seed % 4 == 1)
        _random_meta(rng, level, mp)
    return lp, mp, level


# the kitchens of tests/test_gpu_random_kitchens.py: together they give every plan class the library dispatches on with
# every agent count it has specialised kernels for (tests/test_random_kitchens.py::test_the_device_kitchens_cover_every_plan_class)
DEVICE_KITCHENS = [32, 16, 72, 68, 28, 132, 36, 20, 108, 31, 1, 5, 3, 7, 13, 9, 30, 12, 14, 54, 0, 29, 2, 10,
                   1017, 1033, 1047, 1002, 1042, 1003, 1115, 1142, 1094, 1011, 1019]


def plan_class(t):
    """the library's rule (cz_tables_create) over CompiledTables: packed = n_comp > 0, one computed range, tab_len <= 128,
    even L, V <= 16 and B <= 16; packed plans with <= 32 (observer, slot) pairs take the specialised kernels, 33-64 pairs
    the two-pairs-per-lane writers, everything else the generic kernels and the any-plan writers"""
    A, L = t.num_agents, t.obs_len
    packed = (t.num_comp_slots > 0 and t.num_obs_ranges == 1 and t.obs_table_len <= 128 and L % 2 == 0
              and t.num_variants <= 16 and len(t.recipe_names) <= 16)
    if packed and A * t.num_comp_slots <= 32:
        return "packed32"
    if packed and A * t.num_comp_slots <= 64:
        return "packed64"
    if L % 2:
        return "generic_odd_L" if A % 2 == 0 else "generic_AL_odd"
    return "generic_AL_even"


def warp_group(t):
    """lanes per environment of the warp kernel (cz_tables_create): 16 when every dynamic slot fits half a warp"""
    return 16 if t.num_dyn_slots <= 16 else 32


def kitchen_config(seed):
    """agents, recipes, scheme, end condition and spawn rates of kitchen `seed`"""
    rng = random.Random(10 ** 6 + seed)
    A = 1 + seed % 4 if seed % 8 < 4 else rng.randint(1, 4)
    cfg = dict(A=A, recipes=[BOOK[rng.randrange(len(BOOK))] for _ in range(A)],
               scheme=rng.choice(["scheme1", "scheme3"]), end_all=rng.random() < 0.5, spawn=None)
    if rng.random() < 0.5:
        cfg["spawn"] = dict(agent_respawn_rate=0.3, agent_despawn_rate=0.1 if A > 1 else 0.0, grace_period=1 + seed % 3)
    return cfg


def served_recipes(level):
    """the book recipes whose every node type is always in the kitchen (OPTIONAL objects do not count), with a
    Cutboard for the chopped ingredients and a Blender for the mashed ones: the scripted cook only crashes on them when
    something is out of its reach, not because an ingredient is missing from the level"""
    have = {"Floor", "Counter"}
    for group in ("STATIC_OBJECTS", "DYNAMIC_OBJECTS"):
        for entry in level[group]:
            (name, spec), = entry.items()
            if spec["COUNT"] > 0 and "OPTIONAL" not in spec:
                have.add(name)
    out = []
    for name in BOOK:
        need = set()
        for node in make_recipe(name):
            need.add(node.type)
            if node.cond == "chopped":
                need.add("Cutboard")
            if node.cond == "mashed":
                need.add("Blender")
        if need <= have:
            out.append(name)
    return out
