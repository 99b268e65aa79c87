"""ctypes binding of libcz_b200.so (the C ABI declared in include/cz_b200.h).

There is NO CPU fallback: importing the package works anywhere (so the table compiler and
the host logic can be tested), but creating an environment without the CUDA library or
without a B200 raises.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CZ_B200_LIB") or os.path.join(HERE, "libcz_b200.so")   # override: A/B builds of the same ABI
ABI_VERSION = 2
STEP_AUTO_RESET = 1
STEP_OBS_F32 = 2
STEP_DEVICE_ACTIONS = 4
STEP_KEEP_ALL = 8
STEP_EPISODE_STATS = 16
STEP_COOK_AGENTS = 32
ERR_BITS = {1: "CUTBOARD_NONE", 2: "REMOVE", 4: "SWITCH_LINK", 8: "SPAWN_LOC", 16: "TRUNC_DESPAWN", 32: "OBS_OVERFLOW",
            64: "OFFGRID", 128: "BAD_ID"}

_P = C.c_void_p


class TableDesc(C.Structure):
    _fields_ = ([("abi_version", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
                 ("num_agents", C.c_int32), ("num_recipes", C.c_int32), ("num_dyn_slots", C.c_int32),
                 ("num_static_slots", C.c_int32), ("num_types", C.c_int32), ("num_comp_slots", C.c_int32),
                 ("num_obs_segs", C.c_int32), ("num_obs_ranges", C.c_int32), ("obs_table_len", C.c_int32),
                 ("obs_segs", (C.c_int32 * 3) * 2), ("obs_ranges", (C.c_int32 * 2) * 3),
                 ("obs_len", C.c_int32), ("num_variants", C.c_int32), ("num_layouts", C.c_int32),
                 ("num_book", C.c_int32), ("max_steps", C.c_int32), ("end_all", C.c_int32), ("action_scheme", C.c_int32),
                 ("grace_period", C.c_int32), ("num_switches", C.c_int32), ("num_blocks", C.c_int32),
                 ("reward_node", C.c_double), ("reward_recipe", C.c_double), ("reward_penalty", C.c_double),
                 ("reward_time", C.c_double), ("respawn_rate", C.c_double), ("despawn_rate", C.c_double)]
                + [(n, _P) for n in ("xlut", "ylut", "grid", "static_cells", "scan_order", "special_cells",
                                     "static_masks", "slot_type", "type_flags", "type_base", "type_count",
                                     "comp_slots", "obs_table", "recipe_nodes", "recipe_len", "pool", "default_recipes",
                                     "spawn_x", "spawn_y", "spawn_n", "layout_cum")])


class PolicyDesc(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("num_variants", C.c_int32), ("lists", _P), ("list_len", _P),
                ("reach", _P), ("first_step", _P)]


class StatsDesc(C.Structure):
    _fields_ = [("n_envs", C.c_int32)] + [(n, _P) for n in ("ret", "episode", "open", "last_ret", "last_len", "last_served",
                                                            "last_success", "finished", "totals")]


class CookDesc(C.Structure):
    _fields_ = [("n_envs", C.c_int32), ("k_capacity", C.c_int32)] + \
               [(n, _P) for n in ("agent_mask", "cook_recipes", "actions_taken", "crashed")]


# every symbol include/cz_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "cz_abi_version": (C.c_int, []),
    "cz_last_error": (C.c_char_p, []),
    "cz_launch_count": (C.c_uint64, []),
    "cz_layout_draw": (C.c_uint64, [C.c_uint64, C.c_uint64, C.c_uint64]),
    "cz_layout_index": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint64]),
    "cz_spawn_uniform": (C.c_double, [C.c_uint64] * 5),
    "cz_tables_create": (C.c_int, [C.POINTER(TableDesc), C.c_int, C.POINTER(_P)]),
    "cz_tables_destroy": (C.c_int, [_P]),
    "cz_state_rows": (C.c_int, [_P]),
    "cz_reset": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "cz_layout_ids": (C.c_int, [_P, _P, C.c_int, C.c_uint64, C.c_int64, C.c_uint64, _P]),
    "cz_step": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_uint32, C.c_uint64, C.c_int64,
                          C.c_uint64, _P]),
    "cz_stats_attach": (C.c_int, [_P, C.POINTER(StatsDesc)]),
    "cz_stats_clear": (C.c_int, [_P, _P, C.c_int, _P]),
    "cz_observe": (C.c_int, [_P, _P, _P, C.c_int, _P]),
    "cz_observe_f32": (C.c_int, [_P, _P, _P, C.c_int, _P]),
    "cz_grid_channels": (C.c_int, [_P]),
    "cz_observe_grid": (C.c_int, [_P, _P, _P, C.c_int, _P]),
    "cz_observe_agents": (C.c_int, [_P, _P, C.c_uint32, _P, C.c_uint32, C.c_int, _P]),
    "cz_observe_grid_agents": (C.c_int, [_P, _P, C.c_uint32, _P, C.c_int, _P]),
    "cz_step_pipelined": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_uint32, C.c_uint64, C.c_int64, _P]),
    "cz_pipeline_config": (C.c_int, [_P, C.c_int, C.c_int]),
    "cz_pipeline_wait": (C.c_int, [_P, _P]),
    "cz_pipeline_wait_state": (C.c_int, [_P, _P]),
    "cz_pipeline_reset": (C.c_int, [_P, C.c_int]),
    "cz_pipeline_current": (C.c_int, [_P]),
    "cz_policy_create": (C.c_int, [_P, C.POINTER(PolicyDesc), C.POINTER(_P)]),
    "cz_policy_destroy": (C.c_int, [_P]),
    "cz_policy_config": (C.c_int, [_P, C.c_int]),
    "cz_policy_act": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, _P]),
    "cz_cook_attach": (C.c_int, [_P, _P, C.POINTER(CookDesc)]),
    "cz_random_actions": (C.c_int, [_P, _P, C.c_int, C.c_uint64, C.c_uint64, C.c_int64, _P]),
    "cz_step_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_uint32, C.c_uint64, C.c_int64, _P]),
}

_lib = None


class NativeError(RuntimeError):
    pass


def load_library():
    """dlopen libcz_b200.so; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(f"{LIB_PATH} not found: build it with `python -m cooking_zoo_b200.build` "
                          "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.cz_abi_version() != ABI_VERSION:
        raise NativeError("libcz_b200.so ABI version mismatch; rebuild it")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise NativeError(f"libcz_b200 error {rc}: {load_library().cz_last_error().decode()}")


def make_desc(t):
    """cz_table_desc over the numpy arrays of a CompiledTables (kept alive by the caller)."""
    d = TableDesc()
    d.abi_version = ABI_VERSION
    d.width, d.height, d.num_agents, d.num_recipes = t.width, t.height, t.num_agents, t.num_recipes
    d.num_dyn_slots, d.num_static_slots, d.num_types = t.num_dyn_slots, t.num_static_slots, t.num_types
    d.num_comp_slots, d.obs_len = t.num_comp_slots, t.obs_len
    d.num_obs_segs, d.num_obs_ranges, d.obs_table_len = t.num_obs_segs, t.num_obs_ranges, t.obs_table_len
    for k in range(2):
        for j in range(3):
            d.obs_segs[k][j] = int(t.obs_segs[k, j])
    for k in range(3):
        for j in range(2):
            d.obs_ranges[k][j] = int(t.obs_ranges[k, j])
    d.num_variants, d.num_layouts, d.num_book = t.num_variants, t.num_layouts, len(t.recipe_names)
    d.max_steps, d.end_all, d.grace_period = t.max_steps, t.end_all, t.grace_period
    d.action_scheme = t.action_scheme
    d.num_switches, d.num_blocks = t.num_switches, t.num_blocks
    d.reward_node, d.reward_recipe, d.reward_penalty = t.reward_node, t.reward_recipe, t.reward_penalty
    d.reward_time, d.respawn_rate, d.despawn_rate = t.reward_time, t.respawn_rate, t.despawn_rate
    keep = []
    for name, dtype in (("xlut", np.float64), ("ylut", np.float64), ("grid", np.uint8),
                        ("static_cells", np.uint8), ("scan_order", np.uint8), ("special_cells", np.uint8),
                        ("static_masks", np.uint64), ("slot_type", np.uint8), ("type_flags", np.uint8),
                        ("type_base", np.uint8), ("type_count", np.uint8), ("comp_slots", np.uint32),
                        ("obs_table", np.float64),
                        ("recipe_nodes", np.uint32), ("recipe_len", np.uint8), ("pool", np.uint32),
                        ("default_recipes", np.uint8), ("spawn_x", np.uint8), ("spawn_y", np.uint8),
                        ("spawn_n", np.uint8)):
        arr = np.ascontiguousarray(getattr(t, name), dtype=dtype)
        keep.append(arr)
        setattr(d, name, arr.ctypes.data)
    d.layout_cum = None
    if getattr(t, "layout_cum", None) is not None:
        arr = np.ascontiguousarray(t.layout_cum, dtype=np.uint64)
        keep.append(arr)
        d.layout_cum = arr.ctypes.data
    return d, keep


def make_policy_desc(t, p):
    """cz_policy_desc over the arrays of policy.compile_policy_tables (kept alive by the caller)."""
    d = PolicyDesc()
    d.abi_version, d.num_variants = ABI_VERSION, t.num_variants
    keep = []
    for name, dtype in (("lists", np.uint8), ("list_len", np.uint8), ("reach", np.uint64), ("first_step", np.uint8)):
        arr = np.ascontiguousarray(p[name], dtype=dtype)
        keep.append(arr)
        setattr(d, name, arr.ctypes.data)
    return d, keep
