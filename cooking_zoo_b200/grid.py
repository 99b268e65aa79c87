"""Channel names of the grid observation (include/cz_b200.h, "grid observation").

The grid is u8 [N, A, C, H, W]: per-cell planes of every agent's world, written on the device by cz_observe_grid from
the packed state.  Channel order for observer a: the 7 static kinds in ST_* code order, 5 static states, one count plane
per dynamic type of the meta file (meta order, types without device slots included), chopped / mashed counts of the
choppable / blendable types, on_plate, then one group of 7 planes per agent (group 0 is the observer, then the other
agents in ascending index).  The grid does not encode the order of contents, free flags, grace periods, the clock or
recipe marks.
"""
from . import entities as E

STATIC_KIND_CHANNELS = ("floor", "counter", "cutboard", "blender", "deliversquare", "switch", "block")
STATIC_STATE_CHANNELS = ("cutboard_ready", "blender_ready", "blender_on", "switch_active", "block_walkable")


def grid_channels(tables):
    """Names of the C channels of the grid observation for these compiled tables, in order."""
    types = list(tables.dyn_types)
    flags = [int(f) for f in tables.type_flags]
    names = list(STATIC_KIND_CHANNELS) + list(STATIC_STATE_CHANNELS)
    names += [f"n:{n}" for n in types]
    names += [f"chopped:{n}" for n, f in zip(types, flags) if f & E.TF_CHOP]
    names += [f"mashed:{n}" for n, f in zip(types, flags) if f & E.TF_BLEND]
    names.append("on_plate")
    for g in range(tables.num_agents):
        names += [f"agent{g}"] + [f"agent{g}_facing{o}" for o in range(1, 5)] + [f"agent{g}_holding", f"agent{g}_active"]
    return names
