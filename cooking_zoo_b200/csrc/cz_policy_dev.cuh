// cz_policy_dev.cuh — the scripted cook's decision (CookingAgent.step) as device functions, with two callers:
// cz_policy_kernel (cz_policy.cuh: one lane per environment over shared-memory state columns, stride OSTRIDE; its merge
// instantiation serves CZ_STEP_COOK_AGENTS on the per-step paths) and cz_warp_kernel's COOK instantiation (cz_warp.cuh:
// the environment's slot records in a per-group scratch, stride 1).  Included by cz_kernels.cu before cz_warp.cuh.
//
// CookingAgent.step (cooking_agents/cooking_agent.py:9-122) + BaseAgent helpers (cooking_agents/base_agent.py:49-199) are
// a pure function of the world; the two graph searches over the Floor tiles are host-built tables per static variant
// (cooking_zoo_b200/policy.py, cz_policy.cuh).
#pragma once

struct CzPolicyDev {
  const uint8_t* lists;       // [V][8][64] cells of each static kind in world_objects order
  const uint8_t* list_len;    // [V][8]
  const uint64_t* reach;      // [V][64]
  const uint8_t* first_step;  // [V][64][64]
  int use_env_marks;          // cook i follows recipe i: take the node marks from the state (CZ_POLICY_ENV_MARKS=0: re-evaluate)
};

// CZ_STEP_COOK_AGENTS: the caller-owned buffers of cz_cook_attach and the tables of its policy (n == 0: nothing attached)
struct CzCookDev {
  CzPolicyDev P;
  const uint8_t* agent_mask;    // [n] bit i: agent i acts by the cook
  const uint8_t* cook_recipes;  // [n][A] book index each cook follows, or NULL: recipe i
  uint8_t* actions_taken;       // [k_cap][n][A]
  uint8_t* crashed;             // [n] or NULL
  int n, k_cap;
};

struct PolList {
  const uint8_t* cells;  // static kind: cell list; nullptr for a dynamic type
  int base, n;
};

__device__ __forceinline__ PolList pol_list(const CzDev& T, const CzPolicyDev& P, uint32_t variant, uint32_t node) {
  PolList l;
  l.cells = nullptr;
  l.base = 0;
  l.n = 0;
  if (node & 256u) {
    const uint32_t kind = node & 7u;
    l.cells = P.lists + ((size_t)variant * 8 + kind) * 64;
    l.n = __ldg(P.list_len + variant * 8 + kind);
  } else if ((node & 255u) != 255u) {
    l.base = __ldg(T.type_base + (node & 255u));
    l.n = __ldg(T.type_count + (node & 255u));
  }
  return l;
}

// k-th entry of observation[type name]: false for an empty slot (OPTIONAL object absent, unused Bread twin)
template <int S>
__device__ __forceinline__ bool pol_item(const PolList& l, const uint32_t* o, int k, uint32_t& loc, uint32_t& rec) {
  if (l.cells) {
    loc = __ldg(l.cells + k);
    rec = O_PRESENT;
    return true;
  }
  rec = o[(l.base + k) * S];
  loc = O_XY(rec);
  return (rec & O_PRESENT) != 0;
}

// check_node_conditions (base_agent.py:192-198): unmet conditions of a node on one object (0 or 1)
__device__ __forceinline__ uint32_t pol_unmet(uint32_t cond, uint32_t rec) {
  return cond == 1u ? !(rec & O_CHOP) : (cond == 2u ? !(rec & O_MASH) : 0u);
}

// BaseAgent.distance squared (monotone in the reference's sqrt; all values are small integers)
__device__ __forceinline__ int pol_d2(uint32_t a, uint32_t b) {
  int dx = (int)(a & 7u) - (int)(b & 7u), dy = (int)(a >> 3) - (int)(b >> 3);
  return dx * dx + dy * dy;
}

// BaseAgent.closest (base_agent.py:128-138) over the cells of a static list that pass `keep`:
// first strictly nearest cell reachable from `origin`; -1 if none (the reference then raises).
__device__ __forceinline__ int pol_closest(const CzPolicyDev& P, uint32_t variant, uint32_t kind, uint32_t origin,
                                           uint64_t keep) {
  const uint8_t* cells = P.lists + ((size_t)variant * 8 + kind) * 64;
  const int n = __ldg(P.list_len + variant * 8 + kind);
  const uint64_t ok = keep & __ldg(P.reach + variant * 64 + origin);
  int best = -1, best_d = 1 << 20;
  for (int k = 0; k < n; ++k) {
    const uint32_t c = __ldg(cells + k);
    if (!(ok >> c & 1ull)) continue;
    const int d = pol_d2(origin, c);
    if (d < best_d) {
      best_d = d;
      best = (int)c;
    }
  }
  return best;
}

#define POL_WALK(from, to) ((uint32_t)__ldg(P.first_step + ((size_t)variant * 64 + (from)) * 64 + (to)))

// generic_sequence (base_agent.py:148-190): get food `slot` processed by an appliance of `kind`
// Per-environment masks every cook of the environment shares (built once, by all lanes, before the divergent cook logic:
// inside pol_appliance these loops ran at ~6 active lanes and were a quarter of the kernel's warp instructions).
struct PolEnv {
  uint64_t filled;  // cells whose static object holds something
  uint64_t app[2];  // cells of the Cutboards / Blenders of the layout variant
};

// cells of the Cutboards / Blenders of the layout variant
__device__ __forceinline__ void pol_app_masks(const CzPolicyDev& P, uint32_t variant, PolEnv& pe) {
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const uint32_t kind = j == 0 ? ST_CUTBOARD : ST_BLENDER;
    const uint8_t* apps = P.lists + ((size_t)variant * 8 + kind) * 64;
    const int n_apps = __ldg(P.list_len + variant * 8 + kind);
    uint64_t cells = 0;
    for (int k = 0; k < n_apps; ++k) cells |= 1ull << __ldg(apps + k);
    pe.app[j] = cells;
  }
}

// a slot record whose object lies in a static object: its cell belongs to PolEnv::filled
__device__ __forceinline__ bool pol_fills(uint32_t r) { return (r & O_PRESENT) && O_CK(r) == CK_STATIC; }

// S: stride in words between the slot records of `o` (OSTRIDE in cz_policy_kernel's shared-memory columns, 1 in the warp
// kernel's per-group scratch, which builds `filled` with a group reduction instead)
template <int S>
__device__ __forceinline__ PolEnv pol_env_masks(const CzDev& T, const CzPolicyDev& P, const uint32_t* o, uint32_t variant) {
  PolEnv pe;
  pe.filled = 0;
  for (int k = 0; k < T.D; ++k) {
    const uint32_t r = o[k * S];
    if (pol_fills(r)) pe.filled |= 1ull << O_XY(r);
  }
  pol_app_masks(P, variant, pe);
  return pe;
}

template <int S>
__device__ __forceinline__ uint32_t pol_appliance(const CzDev& T, const CzPolicyDev& P, const PolEnv& pe, const uint32_t* o,
                                                  uint32_t variant, uint32_t agent_rec, uint32_t kind, uint32_t slot, bool& crash) {
  const uint32_t me = A_XY(agent_rec);
  const uint32_t rec = o[slot * S];
  const uint32_t at = O_XY(rec);
  const uint64_t near = __ldg(P.reach + variant * 64 + me);
  const uint64_t app_cells = pe.app[kind == ST_CUTBOARD ? 0 : 1] & near;
  // `obj in appliance.content` for a reachable appliance: walk into it (the bump chops / blends)
  if (O_CK(rec) == CK_STATIC && (app_cells >> at & 1ull)) return POL_WALK(me, at);
  const uint64_t filled = pe.filled;  // static objects with content
  const uint64_t empty_apps = app_cells & ~filled;
  int target;
  if (A_HAS(agent_rec) && A_HOLD(agent_rec) == slot) {
    if (empty_apps) target = pol_closest(P, variant, kind, at, empty_apps);
    else target = pol_closest(P, variant, ST_COUNTER, at, near);
  } else if (empty_apps) {
    if (A_HAS(agent_rec)) target = pol_closest(P, variant, ST_COUNTER, me, near & ~filled);  // put the other thing down
    else return POL_WALK(me, at);
  } else {
    target = pol_closest(P, variant, kind, me, app_cells);
  }
  if (target < 0) {
    crash = true;  // walk_to_location(None): tuple(None) raises (base_agent.py:63)
    return 0;
  }
  return POL_WALK(me, (uint32_t)target);
}

// CookingAgent.step for cook `i` following book recipe `rid`
// `marks`: the node marks of this recipe as the environment's own step left them (CZ_ROW_MARKS; bit k = node k marked), or
// 0x100 when the cook follows a recipe the environment does not score and the graph has to be evaluated here.  The cook
// re-evaluates its private copy of the graph from the same world the environment evaluated after the step
// (cooking_agent.py:12 / cooking_env.py:300, both Recipe.update_recipe_state, recipe.py:77-87), so the marks are the same.
template <int S>
__device__ __forceinline__ uint32_t pol_cook(const CzDev& T, const CzPolicyDev& P, const PolEnv& pe, const uint32_t* o,
                                             uint32_t variant, uint32_t agent_rec, uint32_t rid, uint32_t marks, bool& crash) {
  const uint32_t me = A_XY(agent_rec);
  const int n = __ldg(T.recipe_len + rid);
  int pick = -1;  // find_node (base_agent.py:49-53): first unmarked node from the back of node_list
  if (marks < 0x100u) {
    const uint32_t open_nodes = ~marks & ((1u << n) - 1u);
    pick = open_nodes ? 31 - __clz(open_nodes) : -1;
  } else {
  // own recipe graph, re-evaluated from the world (cooking_agent.py:12, recipe.py:77-87)
  uint64_t m[CZ_MAX_NODES];
#pragma unroll
  for (int k = CZ_MAX_NODES - 1; k >= 0; --k) {
    m[k] = 0;
    if (k < n) {
      const uint32_t node = __ldg(T.recipe_nodes + rid * CZ_MAX_NODES + k);
      uint64_t mask = (node & 256u) ? __ldg(T.static_masks + variant * 8 + (node & 7u))
                                    : cz_node_mask<S>(o, __ldg(T.recipe_spans + rid * CZ_MAX_NODES + k));
      const uint32_t kids = node >> 16;
#pragma unroll
      for (int j = k + 1; j < CZ_MAX_NODES; ++j)
        if (kids & (1u << j)) mask &= m[j];
      m[k] = mask;
      if (!mask && pick < 0) pick = k;
    }
  }
  }
  if (pick < 0) return 0;
  const uint32_t node = __ldg(T.recipe_nodes + rid * CZ_MAX_NODES + pick);
  const uint32_t cond = (node >> 9) & 3u, kids = node >> 16;
  const PolList objs = pol_list(T, P, variant, node);
  const uint64_t near = __ldg(P.reach + variant * 64 + me);

  // ---- compute_condition_action (cooking_agent.py:42-55): the object closest to fulfilling the node
  {
    int best = -1, best_key = 1 << 20;
    uint32_t best_rec = 0;
    for (int k = 0; k < objs.n; ++k) {
      uint32_t loc, rec;
      if (!pol_item<S>(objs, o, k, loc, rec)) continue;
      const int key = (int)(pol_unmet(cond, rec) << 10) + pol_d2(me, loc);  // sorted by (unmet, distance), first wins
      if (key < best_key) {
        best_key = key;
        best = k;
        best_rec = rec;
      }
    }
    if (best < 0) {
      crash = true;  // sorted([])[0] (cooking_agent.py:49)
      return 0;
    }
    if (pol_unmet(cond, best_rec)) {
      // handle_condition_sequence (base_agent.py:133-146): CHOPPED -> Cutboard, MASHED -> Blender
      const uint32_t act = pol_appliance<S>(T, P, pe, o, variant, agent_rec, cond == 1u ? ST_CUTBOARD : ST_BLENDER,
                                         (uint32_t)(objs.base + best), crash);
      if (crash) return 0;
      if (act) return act;
    }
  }

  // ---- compute_contains_action (cooking_agent.py:26-40)
  // get_location_with_most_objects (:99-122)
  int main_cell = -1, main_count = -1;
  for (int k = 0; k < objs.n; ++k) {
    uint32_t mloc, mrec;
    if (!pol_item<S>(objs, o, k, mloc, mrec) || !(near >> mloc & 1ull)) continue;
    int count = 0;
    for (int j = pick + 1; j < n; ++j) {
      if (!(kids >> j & 1u)) continue;
      const uint32_t kid = __ldg(T.recipe_nodes + rid * CZ_MAX_NODES + j);
      if (kid & 256u) {  // static child type (no_recipe's Floor): cells are unique, membership is one mask test
        count += (int)((__ldg(T.static_masks + variant * 8 + (kid & 7u)) & near) >> mloc & 1ull);
        continue;
      }
      const PolList kl = pol_list(T, P, variant, kid);
      for (int q = 0; q < kl.n; ++q) {
        uint32_t loc, rec;
        if (!pol_item<S>(kl, o, q, loc, rec) || !(near >> loc & 1ull)) continue;
        if (loc == mloc && !pol_unmet((kid >> 9) & 3u, rec)) ++count;
      }
    }
    if (count > main_count || (count == main_count && pol_d2(me, mloc) < pol_d2(me, (uint32_t)main_cell))) {
      main_count = count;
      main_cell = (int)mloc;
    }
  }
  // get_best_contains_obj (:57-76): nearest object of any child type that is not already there
  int target = -1, target_d = 1 << 20;
  for (int j = pick + 1; j < n; ++j) {
    if (!(kids >> j & 1u)) continue;
    const uint32_t kid = __ldg(T.recipe_nodes + rid * CZ_MAX_NODES + j);
    if (kid & 256u) {
      // static child type: when the cook stands on such a cell (distance 0, and only that cell is at distance 0) the
      // list walk can only return it, unless an earlier candidate already sits at distance 0
      const uint64_t cells = __ldg(T.static_masks + variant * 8 + (kid & 7u)) & near;
      if ((cells >> me & 1ull) && main_cell >= 0 && (int)me != main_cell) {
        if (0 < target_d) {
          target_d = 0;
          target = (int)me;
        }
        continue;
      }
    }
    const PolList kl = pol_list(T, P, variant, kid);
    for (int q = 0; q < kl.n; ++q) {
      uint32_t loc, rec;
      if (!pol_item<S>(kl, o, q, loc, rec) || !(near >> loc & 1ull)) continue;
      if (main_cell < 0) {
        crash = true;  // None.location (:66)
        return 0;
      }
      if ((int)loc == main_cell) continue;
      const int d = pol_d2(me, loc);
      if (d < target_d) {
        target_d = d;
        target = (int)loc;
      }
    }
  }
  if (target < 0) return 0;
  return ((uint32_t)target == me) ? POL_WALK(me, (uint32_t)main_cell) : POL_WALK(me, (uint32_t)target);
}
