// cz_warp.cuh — ONE WARP PER ENVIRONMENT: the latency-optimised step, persistent over K steps (sm_100a).
//
// The lane-per-environment kernels (cz_device.cuh) walk ~2.4 k dependent instructions per step: right for
// 131072 environments (one instruction stream serves 32 environments), wrong for BASELINE config 3's 4096, where
// a step is bounded by that chain and not by bytes.  Here lane s owns dynamic-object slot s, so every `for slot`
// loop of the dynamics collapses into a ballot / a warp reduction, and agents, static bits, recipe marks and the
// clock are warp-uniform registers.  The whole environment lives in registers across the K steps of one launch:
// state is read once and written once, actions come from a resident [K][n][A] array or from the counter stream of
// cz_random_actions, and the A observation rows leave through the same staging rows / 128-bit stores as
// cz_obs_envs_kernel after every step.
//
// Semantics are those of cz_step_env (cz_device.cuh), statement by statement; citations there and below are to
// /root/reference/cooking_zoo/...  Bit-identity with cz_step x K is tested in tests/test_gpu_ksteps.py.
// Included by cz_kernels.cu (needs BlockSmem, LaneSlot, cz_lane_slot_packed).
#pragma once
#ifndef CZ_WARP_WHOLE
#define CZ_WARP_WHOLE 1  // whole rows staged (table segments by cp.async), one bulk store per environment and step
                        // (config 3, K = 64: 4.33 against 4.44 us per step for CZ_WARP_TMA alone; 0: A/B build)
#endif
#ifndef CZ_WARP_TMA
#define CZ_WARP_TMA 1  // the computed range of the rows leaves through cp.async.bulk (0: lane stores; K = 64: 4.45 vs 4.71 us per step)
#endif

#ifndef WK_WARPS
#define WK_WARPS 4  // environments (warps) per block
#endif
#define WK_FULL 0xffffffffu
#define WK_WORDS 136  // per-warp scratch words: cells[64] | skp[8] | plist[32] (uint2)
#define CZ_ACTION_STREAM 0xA5A5A5A5A5A5A5A5ull  // keeps the action stream apart from the spawn stream of the same seed

// An environment is owned by a GROUP of G lanes (G = 16 when it has at most 16 dynamic slots: two environments per
// warp, every instruction serves both; G = 32 otherwise).  Lane g of the group owns dynamic slot g.  All collectives
// are restricted to the group's lanes (gmask), so the two halves of a warp may diverge freely.
template <int NA, int G>
struct WEnv {
  uint32_t rec;    // this lane's dynamic-object record (0 for lanes >= D)
  uint32_t tf;     // type flags of this lane's slot
  uint32_t rank;   // position of this lane's slot in get_objects_at's scan order (cooking_world.py:232-241)
  uint32_t m_none, m_chop, m_mash;  // (recipe, node) pairs this slot's type can satisfy: always / when chopped / when mashed
  uint32_t ag[NA];                  // agent records (group-uniform)
  uint32_t sbits, tinfo, marks, variant, rids, episode, err;  // group-uniform
  uint32_t pairs_static_only, static_marks;  // pairs whose whole subtree is static, and which of them hold in this variant
  uint32_t n_vote;                           // entries of `plist`
  double v_idle;                             // a recipe's reward on a step that changes none of its marks
  uint64_t walk64, block64;  // cells whose static object is always walkable / is a Block (walkable by state)
  const SmemTabs* st;
  uint32_t* cells;   // [64] per-group scratch: pairs satisfied per cell
  uint32_t* skp;     // [8]  pairs satisfied by a static kind
  uint2* plist;      // [32] {subtree mask, own bit} of every pair that is decided by looking at the objects
  uint32_t gmask;    // the group's lanes
  int g;             // lane within the group = dynamic slot owned by this lane
  int gbase;         // first lane of the group
};

// ---- group collectives -----------------------------------------------------------------------------------------
template <int NA, int G>
__device__ __forceinline__ uint32_t g_ballot(const WEnv<NA, G>& e, bool p) {  // bit s = predicate of the lane owning slot s
  if (G == 32) return __ballot_sync(WK_FULL, p);
  return __ballot_sync(e.gmask, p) >> e.gbase;
}
template <int NA, int G>
__device__ __forceinline__ bool g_any(const WEnv<NA, G>& e, bool p) { return __any_sync(G == 32 ? WK_FULL : e.gmask, p); }
template <int NA, int G>
__device__ __forceinline__ uint32_t g_shfl(const WEnv<NA, G>& e, uint32_t v, int src) {
  return __shfl_sync(G == 32 ? WK_FULL : e.gmask, v, src, G);
}
template <int NA, int G>
__device__ __forceinline__ uint32_t g_max(const WEnv<NA, G>& e, uint32_t v) { return __reduce_max_sync(G == 32 ? WK_FULL : e.gmask, v); }
template <int NA, int G>
__device__ __forceinline__ uint32_t g_or(const WEnv<NA, G>& e, uint32_t v) { return __reduce_or_sync(G == 32 ? WK_FULL : e.gmask, v); }
template <int NA, int G>
__device__ __forceinline__ void g_sync(const WEnv<NA, G>& e) { __syncwarp(G == 32 ? WK_FULL : e.gmask); }

template <int NA>
__device__ __forceinline__ uint32_t wk_sel(const uint32_t (&a)[NA], int i) {
  uint32_t v = a[0];
#pragma unroll
  for (int j = 1; j < NA; ++j)
    if (i == j) v = a[j];
  return v;
}

template <int NA>
__device__ __forceinline__ void wk_put(uint32_t (&a)[NA], int i, uint32_t v) {
#pragma unroll
  for (int j = 0; j < NA; ++j)
    if (i == j) a[j] = v;
}

template <int NA, int G>
__device__ __forceinline__ bool wk_agent_on(const WEnv<NA, G>& e, uint32_t cell) {
  bool on = false;
#pragma unroll
  for (int j = 0; j < NA; ++j)
    if (A_XY(e.ag[j]) == cell) on = true;
  return on;
}

template <int NA, int G>
__device__ __forceinline__ bool wk_walkable(const CzDev& T, const WEnv<NA, G>& e, uint32_t cell) {
  constexpr bool FAST = true;
  const SmemTabs* st = e.st;
  if ((e.walk64 >> cell) & 1ull) return true;
  if ((e.block64 >> cell) & 1ull) return (e.sbits & SB_BLK_WALK(TAB_GRID(e.variant, cell) >> 4)) != 0;
  return false;
}

// Subtree mask of pair p = 8 r + k in pair space (0 when the environment has no such node)
template <int NA, int G>
__device__ __forceinline__ uint32_t wk_pair_desc(const CzDev& T, const WEnv<NA, G>& e, int p) {
  constexpr bool FAST = true;
  const SmemTabs* st = e.st;
  const int r = p >> 3, k = p & 7;
  if (r >= T.R) return 0u;
  const uint32_t rid = (e.rids >> (8 * r)) & 255u;
  return k < (int)TAB_RLEN(rid) ? (uint32_t)st->recipe_desc[rid][k] << (8 * r) : 0u;
}

// everything that depends on the static variant of the current layout (changes only on reset)
template <int NA, int G>
__device__ __forceinline__ void wk_variant_consts(const CzDev& T, WEnv<NA, G>& e) {
  constexpr bool FAST = true;
  const SmemTabs* st = e.st;
  e.walk64 = TAB_SMASK(e.variant, ST_FLOOR) | TAB_SMASK(e.variant, ST_SWITCH);
  e.block64 = TAB_SMASK(e.variant, ST_BLOCK);
  uint32_t* scratch = e.cells;  // rewritten by every step anyway
  if (e.g < T.D) scratch[TAB_SCAN(e.variant, e.g)] = (uint32_t)e.g;
  g_sync(e);
  e.rank = e.g < T.D ? scratch[e.g] : 0u;
  g_sync(e);
  // a node whose whole subtree is static is decided by the variant's static masks alone: one lane decides one pair
  e.static_marks = 0;
#pragma unroll
  for (int p0 = 0; p0 < 32; p0 += G) {
    const int p = p0 + e.g;
    bool holds = false;
    if (e.pairs_static_only >> p & 1u) {
      const int r = p >> 3;
      const uint32_t rid = (e.rids >> (8 * r)) & 255u;
      const uint32_t d = wk_pair_desc(T, e, p) >> (8 * r);
      uint64_t m = ~0ull;
#pragma unroll 1
      for (int j = 0; j < CZ_MAX_NODES; ++j)
        if (d >> j & 1u) m &= TAB_SMASK(e.variant, TAB_RNODE(rid, j) & 7u);
      holds = m != 0;
    }
    e.static_marks |= g_ballot(e, holds) << p0;
  }
}

// (recipe, node) pair p = 8 r + k, the bit layout of the MARKS word.  Per lane: the pairs an object in this slot
// satisfies on its own (type + condition, recipe.py:96-98); per group: the pairs a static kind satisfies, and the
// compact list of pairs that have to be looked for among the objects.  The recipes of an environment never change
// inside a launch, so this runs once.
template <int NA, int G>
__device__ __forceinline__ void wk_recipe_consts(const CzDev& T, WEnv<NA, G>& e) {
  constexpr bool FAST = true;
  const SmemTabs* st = e.st;
  const uint32_t my_type = e.g < T.D ? TAB_STYPE(e.g) : 0xFEu;
  e.m_none = e.m_chop = e.m_mash = 0;
  uint32_t pairs_static = 0;
  if (e.g < 8) e.skp[e.g] = 0;
  g_sync(e);
#pragma unroll 1
  for (int r = 0; r < T.R; ++r) {
    const uint32_t rid = (e.rids >> (8 * r)) & 255u;
    const int n = TAB_RLEN(rid);
#pragma unroll 1
    for (int k = 0; k < n; ++k) {
      const uint32_t node = TAB_RNODE(rid, k), bit = 1u << (8 * r + k);
      if (node & 256u) {
        pairs_static |= bit;
        if (e.g == 0) e.skp[node & 7u] |= bit;
      } else if ((node & 255u) == my_type) {
        const uint32_t cond = (node >> 9) & 3u;
        if (cond == 1u) e.m_chop |= bit;
        else if (cond == 2u) e.m_mash |= bit;
        else e.m_none |= bit;
      }
    }
  }
  e.pairs_static_only = 0;
  e.n_vote = 0;
#pragma unroll
  for (int p0 = 0; p0 < 32; p0 += G) {
    const int p = p0 + e.g;
    const uint32_t d = wk_pair_desc(T, e, p);
    const bool static_only = d != 0 && (d & ~pairs_static) == 0;
    const bool vote = d != 0 && !static_only;
    e.pairs_static_only |= g_ballot(e, static_only) << p0;
    const uint32_t m_vote = g_ballot(e, vote);
    if (vote) e.plist[e.n_vote + __popc(m_vote & ((1u << e.g) - 1u))] = make_uint2(d, 1u << p);
    e.n_vote += __popc(m_vote);
  }
  g_sync(e);
  // reward of a recipe none of whose marks changed: the reference's sum with every term but the time penalty at zero
  double v = 0.0;
  v = __dadd_rn(v, __dmul_rn(0.0, T.r_node));
  v = __dadd_rn(v, 0.0);
  v = __dadd_rn(v, 0.0);
  e.v_idle = __dadd_rn(v, T.r_time);
}

// Recipe.update_recipe_state for every recipe of the environment at once (recipe.py:77-104).  A node is marked iff
// some cell holds, for the node and every descendant, an object that satisfies that node on its own (the AND of the
// children's cell masks in cz_recipe_marks, unrolled over the subtree).  Lanes OR their slot's pairs into a per-cell
// word, read back everything satisfied at their own cell, test every listed pair against it, and one OR-reduction
// collects the marks.
template <int NA, int G>
__device__ __forceinline__ uint32_t wk_recipe_marks(const CzDev& T, WEnv<NA, G>& e) {
  constexpr bool FAST = true;
  const SmemTabs* st = e.st;
  const uint32_t rec = e.rec;
  const bool present = (rec & O_PRESENT) != 0;
  const uint32_t sat = present ? (e.m_none | ((rec & O_CHOP) ? e.m_chop : 0u) | ((rec & O_MASH) ? e.m_mash : 0u)) : 0u;
#pragma unroll
  for (int c = 0; c < 64; c += G) e.cells[c + e.g] = 0;
  g_sync(e);
  if (sat) atomicOr(e.cells + O_XY(rec), sat);
  g_sync(e);
  uint32_t here = 0;
  if (present) here = e.cells[O_XY(rec)] | e.skp[TAB_GRID(e.variant, O_XY(rec)) & 7u];
  uint32_t full = 0;
#pragma unroll 1
  for (uint32_t j = 0; j < e.n_vote; ++j) {
    const uint2 pd = e.plist[j];
    if ((here & pd.x) == pd.x) full |= pd.y;
  }
  g_sync(e);
  return g_or(e, full) | e.static_marks;
}

// Object.move_to / Plate.move_to (abstract_classes.py:21-22, world_objects.py:393-396): slot s and, for a Plate that
// carries items, its content.  `carries` = s is a plate with a non-zero item count.
template <int NA, int G>
__device__ __forceinline__ void wk_move_obj(WEnv<NA, G>& e, uint32_t s, bool carries, uint32_t xy) {
  if ((uint32_t)e.g == s || (carries && O_ON_PLATE(e.rec, s))) e.rec = O_WITH_XY(e.rec, xy);
}

// list.remove(obj) on the content of the static object at `cell`: later items shift down
template <int NA, int G>
__device__ __forceinline__ void wk_remove_from_static(WEnv<NA, G>& e, uint32_t cell, uint32_t pos) {
  if (O_IN_STATIC_AT(e.rec, cell) && O_POS(e.rec) > pos) e.rec -= 1u << 17;
}

// free-flag refresh of one container (cooking_world.py:82-88): last item free, the others not
template <int NA, int G>
__device__ __forceinline__ void wk_refresh_free(WEnv<NA, G>& e, bool in) {
  const uint32_t top = g_max(e, in ? O_POS(e.rec) + 1u : 0u);
  if (in) e.rec = (O_POS(e.rec) + 1u == top) ? (e.rec | O_FREE) : (e.rec & ~O_FREE);
}

// resolve_interaction -> resolve_execute_action | resolve_primary_interaction -> attempt_merge (cz_interact)
template <int NA, int G>
__device__ __forceinline__ uint32_t wk_interact(const CzDev& T, WEnv<NA, G>& e, const int i, uint32_t cell, uint32_t mode, bool& stale) {
  // `i` is a run-time index: the caller's agent loop stays rolled so that this body exists once (code size)
  constexpr bool FAST = true;
  const SmemTabs* st = e.st;
  const int lane = e.g;  // slot owned by this lane
  const uint32_t agent_rec = wk_sel(e.ag, i);
  const uint32_t g = TAB_GRID(e.variant, cell);
  const uint32_t kind = g & 15u, sp = g >> 4;
  // the objects at the faced cell, in scan order (cooking_world.py:232-241)
  const bool at = O_AT(e.rec, cell);
  const uint32_t m_at = g_ballot(e, at);
  const int n_dyn = __popc(m_at);
  const uint32_t m_plate = g_ballot(e, at && (e.tf & TF_PLATE));
  const int n_plates = __popc(m_plate);
  const int plate = n_plates ? 31 - __clz(m_plate) : -1;  // only used when there is exactly one
  const bool any_not_done = g_any(e, at && !(e.tf & TF_PLATE) && !(e.rec & (O_CHOP | O_MASH)));
  const int n_content = __popc(g_ballot(e, at && O_CK(e.rec) == CK_STATIC));
  const uint32_t k_last = g_max(e, at ? ((e.rank << 5) | (uint32_t)lane) + 1u : 0u);
  const uint32_t k_free = g_max(e, (at && (e.rec & O_FREE)) ? (((63u - e.rank) << 5) | (uint32_t)lane) + 1u : 0u);
  const int last = k_last ? (int)((k_last - 1u) & 31u) : -1;
  const int first_free = k_free ? (int)((k_free - 1u) & 31u) : -1;
  const bool blocked = wk_agent_on(e, cell);

  if (mode == 6u) {
    // ---- resolve_interaction_pick_up_special (cooking_world.py:138-154)
    if (blocked || A_HAS(agent_rec) || n_dyn == 0 || n_plates != 1) return 0xFFu;
    const uint32_t k_top = g_max(e, O_ON_PLATE(e.rec, plate) ? ((O_POS(e.rec) << 5) | (uint32_t)lane) + 1u : 0u);
    if (!k_top) return 0xFFu;
    const int ts = (int)((k_top - 1u) & 31u);
    if (lane == plate) e.rec -= O_PCOUNT_ONE;
    if (lane == ts) e.rec = O_WITH_XY(O_WITH_CONT(e.rec, CK_HELD, i, 0), A_XY(agent_rec));
    wk_put(e.ag, i, (agent_rec & ~(0x3Fu << 9)) | (1u << 9) | ((uint32_t)ts << 10));
    return (uint32_t)plate;
  }
  if (mode == 7u || (mode == 0u && (kind == ST_CUTBOARD || kind == ST_BLENDER) && any_not_done)) {
    // ---- resolve_execute_action (cooking_world.py:156-170)
    if (blocked) return 0xFFu;
    if (kind != ST_CUTBOARD && kind != ST_BLENDER) return 0xFFu;
    if (kind == ST_CUTBOARD) {  // Cutboard.action (world_objects.py:250-269)
      if (!(e.sbits & SB_CUT_READY(sp))) return 0xFFu;
      for (int p = 0; p < n_content; ++p) {
        const uint32_t m = g_ballot(e, O_IN_STATIC_AT(e.rec, cell) && O_POS(e.rec) == (uint32_t)p);
        if (!m) break;
        const int s = 31 - __clz(m);
        const uint32_t r = g_shfl(e, e.rec, s);
        const uint32_t tf = g_shfl(e, e.tf, s);
        if (!(tf & TF_CHOP)) return 0xFFu;
        if (r & O_CHOP) continue;
        if (lane == s) e.rec = r | O_CHOP;
        e.sbits &= ~SB_CUT_READY(sp);
        if (tf & TF_SPAWN) {  // Bread.chop spawns a chopped twin (world_objects.py:738-745)
          const uint32_t tid = TAB_STYPE(s);
          const int base = TAB_TBASE(tid), cnt = TAB_TCOUNT(tid);
          const uint32_t m_free = g_ballot(e, lane >= base && lane < base + cnt && !(e.rec & O_PRESENT));
          if (!m_free) {
            e.err |= CZ_ERR_OBS_OVERFLOW;
          } else {
            if (lane == __ffs(m_free) - 1) e.rec = O_WITH_CONT(cell | O_PRESENT | O_CHOP | O_FREE, CK_STATIC, 0, n_content);
            stale = true;
          }
        }
        return 0xFFu;
      }
      e.err |= CZ_ERR_CUTBOARD_NONE;
    } else {  // Blender.action (world_objects.py:356-360)
      if (e.sbits & SB_BL_READY(sp)) e.sbits ^= SB_BL_TOGGLE(sp);
    }
    return 0xFFu;
  }

  // ---- resolve_primary_interaction (cooking_world.py:114-136)
  if (blocked) return 0xFFu;
  const uint32_t axy = A_XY(agent_rec);
  if (!A_HAS(agent_rec)) {
    if (n_dyn == 0) return 0xFFu;
    bool rel = true;  // StaticObject.releases() with side effects
    if (kind == ST_DELIVER) rel = false;
    else if (kind == ST_CUTBOARD) {
      if (n_content == 1) e.sbits &= ~SB_CUT_READY(sp);
    } else if (kind == ST_BLENDER) {
      if (e.sbits & SB_BL_TOGGLE(sp)) rel = false;
      else if (n_content - 1 == 0) e.sbits &= ~SB_BL_READY(sp);
    }
    if (!rel) return 0xFFu;
    const int gs = first_free >= 0 ? first_free : last;
    const uint32_t r = g_shfl(e, e.rec, gs);
    const uint32_t gtf = g_shfl(e, e.tf, gs);
    if (O_CK(r) != CK_STATIC) return 0xFFu;  // `object_to_grab in static_object.content`
    if (n_content > 1) {
      wk_remove_from_static(e, cell, O_POS(r));
      stale = true;
    }
    if (lane == gs) e.rec = O_WITH_CONT(r, CK_HELD, i, 0);
    wk_move_obj(e, (uint32_t)gs, (gtf & TF_PLATE) && O_PCOUNT(r), axy);  // Agent.grab (world_objects.py:786-788)
    wk_put(e.ag, i, (agent_rec & ~(0x3Fu << 9)) | (1u << 9) | ((uint32_t)gs << 10));
    return 0xFFu;
  }

  // ---- attempt_merge (cooking_world.py:243-261)
  const uint32_t h = A_HOLD(agent_rec);
  const uint32_t hr = g_shfl(e, e.rec, h);
  const uint32_t htf = g_shfl(e, e.tf, h);
  const uint32_t dropped = agent_rec & ~(0x3Fu << 9);
  if (n_plates == 1) {
    if ((htf & (TF_CHOP | TF_BLEND)) && (hr & (O_CHOP | O_MASH))) {  // Plate.accepts (world_objects.py:408-409)
      const uint32_t n = O_PCOUNT(g_shfl(e, e.rec, plate));
      if (n < 64) {
        if (n && O_ON_PLATE(e.rec, plate)) e.rec &= ~O_FREE;
        if (lane == plate) e.rec += O_PCOUNT_ONE;
        if (lane == (int)h) e.rec = O_WITH_XY(O_WITH_CONT(hr, CK_PLATE, plate, n) | O_FREE, cell);
        wk_put(e.ag, i, dropped);
      }
    }
  } else if ((htf & TF_PLATE) && n_dyn > 0) {
    const uint32_t pr = g_shfl(e, e.rec, last);
    const uint32_t ptf = g_shfl(e, e.tf, last);
    if ((ptf & (TF_CHOP | TF_BLEND)) && (pr & (O_CHOP | O_MASH))) {
      const uint32_t n = O_PCOUNT(hr);
      if (n < 64) {
        if (n && O_ON_PLATE(e.rec, h)) e.rec &= ~O_FREE;
        if (lane == (int)h) e.rec = hr + O_PCOUNT_ONE;
        if (O_CK(pr) == CK_STATIC) {
          if (n_content > 1) {
            wk_remove_from_static(e, cell, O_POS(pr));
            stale = true;
          }
        } else {
          e.err |= CZ_ERR_REMOVE;
        }
        if (lane == last) e.rec = O_WITH_XY(O_WITH_CONT(pr, CK_PLATE, h, n) | O_FREE, axy);
      }
    }
  } else {
    bool ok = false;  // StaticObject.accepts
    if (kind == ST_COUNTER || kind == ST_DELIVER) ok = n_content < 1;
    else if (kind == ST_CUTBOARD) ok = (htf & TF_CHOP) && n_content < 1 && !(hr & O_CHOP);
    else if (kind == ST_BLENDER)
      ok = (htf & TF_BLEND) && !(e.sbits & SB_BL_TOGGLE(sp)) && n_content + 1 <= 1 && !(hr & O_MASH);
    if (ok) {
      if (kind == ST_CUTBOARD) e.sbits |= SB_CUT_READY(sp);
      if (kind == ST_BLENDER) e.sbits |= SB_BL_READY(sp);
      if (lane == (int)h) e.rec = O_WITH_CONT(hr, CK_STATIC, 0, n_content) | O_FREE;
      wk_move_obj(e, h, (htf & TF_PLATE) && O_PCOUNT(hr), cell);
      wk_put(e.ag, i, dropped);
    }
  }
  return 0xFFu;
}

// CookingEnvironment.accumulated_step (cooking_env.py:243-269) for the group's environment (cz_step_env), or, when
// `fresh` is set, only the recipe evaluation of a state that was just re-initialised (auto-reset): both paths share the
// one inlined copy of wk_recipe_marks.  rw / te / tr: reward, terminated, truncated of every agent (group-uniform).
// Agent loops stay rolled (`#pragma unroll 1`, agents picked with wk_sel / wk_put) and wk_interact has one call site:
// the step is bound by instruction fetch, so the size of the loop body is what counts (profiles/r02_notes.md).
template <int NA, int G>
__device__ __forceinline__ void wk_step_env(const CzDev& T, WEnv<NA, G>& e, const uint32_t act_packed, const bool fresh,
                                            double (&rw)[NA], uint32_t& term_mask, uint32_t& trunc_out, uint64_t seed,
                                            uint64_t genv) {
  constexpr bool FAST = true;
  constexpr int A = NA;
  const SmemTabs* st = e.st;
  const bool scheme1 = T.scheme == 1;
  const uint32_t t = TI_T(e.tinfo) + 1;
  uint32_t active = 0, changed = 0, relevant = 0, trunc_mask = 0;
  bool time_up = false;
  if (!fresh) {
#pragma unroll
  for (int i = 0; i < A; ++i)
    if (A_ACTIVE(e.ag[i])) active |= 1u << i;

  // ---- action_scheme3.perform_agent_actions (action_scheme3.py:4-16)
  uint32_t apack = 0, fpack = 0, epack = 0x80808080u;
#pragma unroll 1
  for (int i = 0; i < A; ++i) {
    if (!(active >> i & 1u)) continue;
    uint32_t ai = (act_packed >> (8 * i)) & 255u;
    if (ai > (scheme1 ? 7u : 4u)) ai = 0;
    uint32_t rec = wk_sel(e.ag, i);
    const int x = rec & 7u, y = (rec >> 3) & 7u;
    uint32_t faced = A_XY(rec);
    if (ai >= 1u && ai <= 4u) {
      rec = (rec & ~(7u << 6)) | (ai << 6);
      wk_put(e.ag, i, rec);
      const int tx = x + (ai == 2) - (ai == 1), ty = y + (ai == 3) - (ai == 4);
      if (tx < 0 || ty < 0 || tx > T.W - 1 || ty > T.H - 1) ai = 0;
      else faced = (uint32_t)(tx | ty << 3);
    }
    const uint32_t tgt = (ai >= 1u && ai <= 4u) ? faced : A_XY(rec);
    const bool w = wk_walkable(T, e, tgt);
    const uint32_t endc = (w ? tgt : A_XY(rec)) | (w ? 0x40u : 0u);
    apack |= ai << (8 * i);
    fpack |= faced << (8 * i);
    epack = (epack & ~(0xFFu << (8 * i))) | (endc << (8 * i));
  }
  uint32_t cancel = 0;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    const uint32_t ei = (epack >> (8 * i)) & 255u;
    if (!(ei & 0x40u) || (ei & 0x80u)) continue;
#pragma unroll
    for (int j = 0; j < A; ++j) {
      const uint32_t ej = (epack >> (8 * j)) & 255u;
      if (j != i && !(ej & 0x80u) && (ej & 63u) == (ei & 63u)) cancel |= 1u << i;
    }
  }
  uint32_t pressed = 0, dirty = 0xFFFFFFFFu, dirty_plate = 0xFFFFFFFFu;
#pragma unroll 1
  for (int i = 0; i < A; ++i) {
    if (!(active >> i & 1u)) continue;
    uint32_t rec = wk_sel(e.ag, i);
    const uint32_t ai = (cancel >> i & 1u) ? 0u : ((apack >> (8 * i)) & 255u);
    uint32_t cell = 0, mode = 0;
    bool interact = false;
    if (scheme1) {
      if (ai == 0u) continue;
      if (ai >= 5u) {
        const uint32_t o = A_ORI(rec);
        const int fx = (int)(rec & 7u) + (o == 2) - (o == 1), fy = (int)((rec >> 3) & 7u) + (o == 3) - (o == 4);
        if (fx < 0 || fy < 0 || fx > T.W - 1 || fy > T.H - 1) {  // IndexError at cooking_world.py:119 / :160; pick-up-special (:138-154) finds nothing
          if (ai != 6u) e.err |= CZ_ERR_OFFGRID;
          continue;
        }
        cell = (uint32_t)(fx | fy << 3);
        mode = ai;
        interact = true;
      }
    }
    if (!interact) {
      const uint32_t tgt = ai ? ((fpack >> (8 * i)) & 63u) : A_XY(rec);
      if (wk_walkable(T, e, tgt)) {  // resolve_walking_action (action_scheme3.py:26-34)
        rec = (rec & ~63u) | tgt;
        wk_put(e.ag, i, rec);
        if (A_HAS(rec)) {  // Agent.move_to (world_objects.py:793-796): the held object and a held plate's content follow
          const uint32_t h = A_HOLD(rec);
          if ((uint32_t)e.g == h || O_ON_PLATE(e.rec, h)) e.rec = O_WITH_XY(e.rec, tgt);
        }
        const uint32_t gk = TAB_GRID(e.variant, tgt);
        if ((gk & 15u) == ST_SWITCH) {
          e.sbits ^= SB_SW_ACTIVE(gk >> 4);
          pressed |= 1u << (gk >> 4);
        }
      } else if (ai && !scheme1) {
        cell = tgt;
        interact = true;
      }
    }
    if (interact) {
      bool stale = false;
      const uint32_t p = wk_interact(T, e, i, cell, mode, stale);  // p != 0xFF only for scheme1's pick-up-special
      if (stale) dirty = (dirty & ~(0xFFu << (8 * i))) | (cell << (8 * i));
      dirty_plate = (dirty_plate & ~(0xFFu << (8 * i))) | (p << (8 * i));
    }
  }

  // ---- progress_world (cooking_world.py:77-88)
  if (e.sbits & (0xFu << 8)) {
    for (int k = 0; k < CZ_MAX_SPECIAL; ++k) {
      if (!(e.sbits & SB_BL_TOGGLE(k))) continue;
      const uint32_t cell = TAB_SPECIAL(e.variant, 1, k);
      if (cell == 0xFFu) continue;
      const bool in = O_IN_STATIC_AT(e.rec, cell);
      if (in && !(e.rec & (O_CHOP | O_MASH))) e.rec |= O_MASH;  // BlenderFood.blend (abstract_classes.py:266-273)
      const bool any_in = g_any(e, in);
      const bool unmashed = g_any(e, in && !(e.rec & O_MASH));
      if (any_in && !unmashed) e.sbits &= ~(SB_BL_TOGGLE(k) | SB_BL_READY(k));
    }
  }
  if (dirty != 0xFFFFFFFFu) {
#pragma unroll
    for (int i = 0; i < A; ++i) {
      const uint32_t c = (dirty >> (8 * i)) & 255u;
      if (c != 0xFFu) wk_refresh_free(e, O_IN_STATIC_AT(e.rec, c));
    }
  }
  if (dirty_plate != 0xFFFFFFFFu) {
#pragma unroll
    for (int i = 0; i < A; ++i) {
      const uint32_t p = (dirty_plate >> (8 * i)) & 255u;
      if (p != 0xFFu) wk_refresh_free(e, O_ON_PLATE(e.rec, p));
    }
  }
  // ---- resolve_linked_interactions (cooking_world.py:90-92)
  if (pressed) {
    uint32_t blocks = 0, n_sw = 0;
    for (int k = 0; k < CZ_MAX_SPECIAL; ++k) {
      if (TAB_SPECIAL(e.variant, 3, k) != 0xFFu) blocks |= SB_BLK_WALK(k);
      if (TAB_SPECIAL(e.variant, 2, k) != 0xFFu) ++n_sw;
    }
    if (n_sw > 1) e.err |= CZ_ERR_SWITCH_LINK;
    for (int k = 0; k < CZ_MAX_SPECIAL; ++k)
      if (pressed >> k & 1u) e.sbits ^= blocks;
  }
  // ---- handle_agent_spawn (cooking_world.py:267-277)
  if (T.respawn > 0.0 || T.despawn > 0.0) {
    uint32_t c = 0;
#pragma unroll 1
    for (int i = 0; i < A; ++i) {
      const uint32_t rec = wk_sel(e.ag, i);
      if (A_GRACE(rec) > 0) { wk_put(e.ag, i, rec - (1u << 16)); continue; }
      const bool act_i = active >> i & 1u;
      if (__popc(active) > 1 && act_i) {
        if (cz_uniform(seed, genv, e.episode, t, c++) < T.despawn) {
          if (!A_HAS(rec)) {
            active &= ~(1u << i);
            changed |= 1u << i;
          }
        }
      } else if (!act_i) {
        if (cz_uniform(seed, genv, e.episode, t, c++) < T.respawn) {
          active |= 1u << i;
          changed |= 1u << i;
          const int nx = __ldg(T.spawn_n + 2 * i), ny = __ldg(T.spawn_n + 2 * i + 1);
          uint32_t cell = A_XY(rec);
          bool found = false;
          #pragma unroll 1
          for (int tries = 0; tries < 1002 && !found; ++tries) {  // parsing.generate_location :154-167
            const int x = __ldg(T.spawn_x + 8 * i + min(nx - 1, (int)(cz_uniform(seed, genv, e.episode, t, c++) * nx)));
            const int y = __ldg(T.spawn_y + 8 * i + min(ny - 1, (int)(cz_uniform(seed, genv, e.episode, t, c++) * ny)));
            const uint32_t cand = (uint32_t)(x | y << 3);
            if (x < T.W && y < T.H && (TAB_GRID(e.variant, cand) & 15u) == ST_FLOOR && !wk_agent_on(e, cand)) {
              cell = cand;
              found = true;
            }
          }
          if (!found) e.err |= CZ_ERR_SPAWN_LOC;
          wk_put(e.ag, i, (rec & 0xFFC0u) | cell | ((uint32_t)T.grace << 16));
        }
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < A; ++i)
      if (A_GRACE(e.ag[i]) > 0) e.ag[i] -= 1u << 16;
  }

  relevant = active | changed;

  // ---- compute_rewards / compute_truncated (cooking_env.py:290-350)
  time_up = t >= (uint32_t)T.max_steps;
  if (time_up) {
    if (TI_NLIVE(e.tinfo) < (uint32_t)A) e.err |= CZ_ERR_TRUNC_DESPAWN;
    trunc_mask = relevant;
    changed = relevant;
    active = 0;
  }
  trunc_mask |= changed & ~active & relevant;
  relevant = active | changed;
  }  // !fresh
  const uint32_t new_marks = wk_recipe_marks(T, e);
#pragma unroll
  for (int i = 0; i < A; ++i) rw[i] = 0.0;
  term_mask = 0;
  trunc_out = 0;
  if (fresh) {  // CookingEnvironment.reset evaluates the recipes once (cooking_env.py:197-198); no step, outputs are zero
    e.marks = new_marks;
    return;
  }
  bool all_done = true, any_done = false;
  if (new_marks == e.marks) {
    // the common step: no node changed, so every recipe's reward is the idle value (bit-identical to the sum below
    // with delta = bonus = malus = 0) and completion is read off the root bits
    const uint32_t roots = 0x01010101u & (T.R >= 4 ? 0xFFFFFFFFu : ((1u << (8 * T.R)) - 1u));
    all_done = (new_marks & roots) == roots;
    any_done = (new_marks & roots) != 0;
#pragma unroll
    for (int i = 0; i < A; ++i)
      if (relevant >> i & 1u) rw[i] = e.v_idle;  // entries beyond the recipe list are cleared below
  } else {
#pragma unroll 1
    for (int r = 0; r < T.R; ++r) {
      const uint32_t before = (e.marks >> (8 * r)) & 255u;
      const uint32_t after = (new_marks >> (8 * r)) & 255u;
      const bool was = before & 1u, now = after & 1u;
      const int delta = __popc(after) - __popc(before);
      double v = 0.0;
      v = __dadd_rn(v, __dmul_rn((double)delta, T.r_node));
      v = __dadd_rn(v, (now && !was) ? T.r_recipe : 0.0);
      v = __dadd_rn(v, (!now && was) ? T.r_penalty : 0.0);
      v = __dadd_rn(v, T.r_time);
      all_done = all_done && now;
      any_done = any_done || now;
      uint32_t m = relevant;  // the r-th relevant agent receives entry r of the recipe lists (cooking_env.py:250-262)
#pragma unroll 1
      for (int q = 0; q < r; ++q) m &= m - 1;
      if (m) {
        const int who = __ffs(m) - 1;
#pragma unroll
        for (int i = 0; i < A; ++i)
          if (i == who) rw[i] = v;
      }
    }
  }
  e.marks = new_marks;
  const bool done = T.end_all ? all_done : any_done;
  int k = 0;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    const bool rel = relevant >> i & 1u;
    if (!rel || k >= T.R) rw[i] = 0.0;
    if (rel) ++k;
    if (rel && done) term_mask |= 1u << i;
    e.ag[i] = (e.ag[i] & ~(1u << 15)) | ((active >> i & 1u) << 15);
  }
  trunc_out = trunc_mask;
  const uint32_t n_live = __popc(relevant);
  e.tinfo = (t & 0xFFFFFu) | ((done || time_up) ? TI_DONE : 0u) | (n_live << 21);
}

// [x, y, flags..., 1] of one (observer, slot) pair into its staging row (cz_pair_store, with the state in registers).
// `pm`: 0-11 row offset | 12-14 features after x,y | 15-16 kind | 17-24 index | 25-26 observer; `live`: the pair exists.
template <int NA, int G>
__device__ __forceinline__ void wk_pair_store(const CzDev& T, const WEnv<NA, G>& e, uint32_t pm, bool live, const double* sxl,
                                              const double* syl, double2* stage, int stage2, int lo) {
  constexpr bool FAST = true;
  const SmemTabs* st = e.st;
  const uint32_t flen = (pm >> 12) & 7u, kind = (pm >> 15) & 3u, idx = (pm >> 17) & 255u;
  const int observer = (int)((pm >> 25) & 3u);
  // every lane of the group takes part in the shuffle; idle lanes read slot 0
  const uint32_t dyn = g_shfl(e, e.rec, (int)(idx & (uint32_t)(G - 1)));
  if (!live) return;
  const bool is_agent = kind == 2, is_static = kind == 0;
  uint32_t rec = is_agent ? wk_sel(e.ag, (int)idx) : dyn;
  uint32_t static_fb = 0;
  if (is_static) {  // live Switch / Block (world_objects.py:174,221)
    const uint32_t cell = TAB_SCELL(e.variant, idx);
    rec = cell != 0xFFu ? (cell | O_PRESENT) : 0u;
    const uint32_t gk = TAB_GRID(e.variant, rec & 63u);
    static_fb = ((gk & 15u) == ST_SWITCH ? (e.sbits >> (12 + (gk >> 4))) : (e.sbits >> (16 + (gk >> 4)))) & 1u;
  }
  const uint32_t me = wk_sel(e.ag, observer);
  const bool present = is_agent || (rec & O_PRESENT);
  const uint32_t c = (rec >> 7) & 1u, m = (rec >> 8) & 1u;
  const uint32_t fb4 = is_static ? static_fb : (is_agent ? ((1u << A_ORI(rec)) >> 1) : (((c | m) ^ 1u) | c << 1 | m << 2));
  const uint32_t one = 1u << (flen - 1);
  const uint32_t fb = present ? ((fb4 & (one - 1u)) | one) : 0u;
  const bool self = is_agent && (int)idx == observer;
  const int x = rec & 7u, y = (rec >> 3) & 7u;
  double X = sxl[x - (self ? 0 : (int)(me & 7u))];
  double Y = syl[y - (self ? 0 : (int)((me >> 3) & 7u))];
  if (!present) { X = 0.0; Y = 0.0; }
  double* out = reinterpret_cast<double*>(stage + observer * stage2) + ((int)(pm & 0xFFFu) - lo);  // lo: row element at stage[0]
  out[0] = X;
  out[1] = Y;
#pragma unroll
  for (int k = 0; k < 5; ++k)
    if (k < (int)flen) *reinterpret_cast<uint2*>(out + 2 + k) = make_uint2(0u, (fb >> k & 1u) ? 0x3FF00000u : 0u);
}

__host__ __device__ inline size_t wk_smem_bytes(int V, int A, int stage_len, int G) {
  const int groups = WK_WARPS * 32 / G;
  return cz_block_smem_head(V) + 64 * 4 + (size_t)groups * (WK_WORDS * 4 + (size_t)A * ((stage_len + 1) / 2) * 16);
}

// STATS (CZ_STEP_EPISODE_STATS): the episode-statistics record of the group's environment (cz_stats.cuh) is loaded in the
// prologue, updated by cz_stats_rule after every step and written in the epilogue next to the state; lane g < NA holds
// agent g's running return, and K steps stay one launch.  STATS = false compiles to the kernel without any of it (the same
// SASS as a kernel without the statistics code); the true instantiation has its own bound for 32-lane groups, where the plain
// kernel's 7 blocks per SM (72 registers) spill the record.
#ifndef CZ_WARP_STATS_MIN_BLOCKS32
#define CZ_WARP_STATS_MIN_BLOCKS32 6
#endif
template <int NA, int G, bool STATS>
__global__ void __launch_bounds__(32 * WK_WARPS, G == 32 ? (STATS ? CZ_WARP_STATS_MIN_BLOCKS32 : 7) : 4)
cz_warp_kernel(const __grid_constant__ CzDev T, uint32_t* __restrict__ state, const uint8_t* __restrict__ actions,
               double* __restrict__ obs, double* __restrict__ reward, uint8_t* __restrict__ term, uint8_t* __restrict__ trunc,
               uint32_t* __restrict__ errflags, int n_envs, int k_steps, uint32_t flags, uint64_t seed, int64_t env_offset,
               uint64_t action_step, const __grid_constant__ CzStatsDev S) {
  constexpr bool FAST = true;
  constexpr int GROUPS = WK_WARPS * 32 / G;  // environments per block
  constexpr int TK = 64 / G;                 // table elements (double2) of a row per lane, at most
  extern __shared__ __align__(16) unsigned char smem_wk[];
  const int lane = threadIdx.x & 31;
  const int g = lane & (G - 1), gbase = lane & ~(G - 1);
  const int grp = (int)(threadIdx.x >> 5) * (32 / G) + (lane >> (G == 32 ? 5 : 4));
  const int env = blockIdx.x * GROUPS + grp;
  BlockSmem* bs = reinterpret_cast<BlockSmem*>(smem_wk);
  const size_t head = cz_block_smem_head(T.V);
  // everything that comes from global memory and does not depend on the block image is requested first, so that the
  // state, the first step's actions and the image arrive in one round trip instead of three (a single-step launch is
  // mostly prologue)
  const bool live = env < n_envs;
  const size_t N = (size_t)n_envs;
  const int D = T.D;
  const uint32_t rec0 = (live && g < D) ? __ldg(state + (size_t)g * N + env) : 0u;
  const uint32_t misc0 = (live && g < NA + CZ_NUM_MISC_ROWS) ? __ldg(state + (size_t)(D + g) * N + env) : 0u;
  uint32_t a_next = (live && actions && g < NA) ? actions[(size_t)env * NA + g] : 0u;
  for (int i = threadIdx.x; i < (int)(head / 16); i += 32 * WK_WARPS)
    reinterpret_cast<uint4*>(bs)[i] = __ldg(reinterpret_cast<const uint4*>(T.blob) + i);
  // (observer, slot) pairs of a row set: one word each, shared by the block
  uint32_t* pmap = reinterpret_cast<uint32_t*>(smem_wk + head);
  const int n_pairs = NA * T.n_comp;
  if (threadIdx.x < 64) {
    const int4 lm = __ldg(T.lane_map + threadIdx.x);
    pmap[threadIdx.x] = lm.x >= 0 ? ((uint32_t)lm.x & 0x1FFFFFFu) | ((uint32_t)lm.y << 25) : 0u;
  }
  const int stage2 = CZ_WARP_WHOLE ? (T.L >> 1) : ((T.stage_len + 1) >> 1);  // double2 per staging row (whole rows or the computed span)
  unsigned char* gsm = smem_wk + head + 256 + (size_t)grp * (WK_WORDS * 4 + (size_t)NA * stage2 * 16);
  uint32_t* wwords = reinterpret_cast<uint32_t*>(gsm);  // cells[64] | skp[8] | plist[32] uint2
  double2* stage = reinterpret_cast<double2*>(gsm + WK_WORDS * 4);
#pragma unroll 1
  for (int k = g; k < NA * stage2; k += G) stage[k] = make_double2(0.0, 0.0);  // never-occupied slots stay zero
  __syncthreads();
  if (!live) return;

  const SmemTabs* st = &bs->tabs;
  const double* sxl = bs->xlut + (T.W - 1);
  const double* syl = bs->ylut + (T.H - 1);
  const int L2 = T.L >> 1, tab2 = T.tab_len >> 1;
  const uint64_t genv = (uint64_t)(env_offset + env);

  WEnv<NA, G> e;
  e.st = st;
  e.g = g;
  e.gbase = gbase;
  e.gmask = G == 32 ? WK_FULL : (0xFFFFu << gbase);
  e.cells = wwords;
  e.skp = wwords + 64;
  e.plist = reinterpret_cast<uint2*>(wwords + 72);
  e.err = 0;
  // ---- state -> registers: lane g holds slot g; agents and the misc words are broadcast inside the group
  e.rec = rec0;
  e.tf = g < D ? TAB_TF(g) : 0u;
  {
    const uint32_t w = misc0;
#pragma unroll
    for (int i = 0; i < NA; ++i) e.ag[i] = g_shfl(e, w, i);
    e.sbits = g_shfl(e, w, NA + CZ_ROW_SBITS);
    e.tinfo = g_shfl(e, w, NA + CZ_ROW_TINFO);
    e.marks = g_shfl(e, w, NA + CZ_ROW_MARKS);
    e.variant = g_shfl(e, w, NA + CZ_ROW_VARIANT);
    e.rids = g_shfl(e, w, NA + CZ_ROW_RECIPES);
    e.episode = g_shfl(e, w, NA + CZ_ROW_EPISODE);
  }
  wk_recipe_consts(T, e);
  wk_variant_consts(T, e);
  // episode statistics: the record, and what the finished episodes of this launch add to it (group-uniform except the
  // returns, which lane g < NA holds for agent g)
  uint32_t st_seen = 0, st_open = 0, st_n = 0, st_len = 0, st_served = 0, st_succ = 0;
  uint32_t st_last = 0;  // the last finished episode: t | served << 20 | success << 28
  double st_ret[1] = {0.0}, st_sum = 0.0, st_lret = 0.0;
  if constexpr (STATS) {
    st_seen = S.episode[env];
    st_open = S.open[env];
    if (g < NA) st_ret[0] = S.ret[(size_t)env * NA + g];
  }

  // where this lane's table elements (double2 units g, g + G, ...) land in a row: segment 0 first, then segment 1
  int tdst[TK];
  {
    const int n0 = T.n_segs > 0 ? T.segs[0][1] >> 1 : 0, n1 = T.n_segs > 1 ? T.segs[1][1] >> 1 : 0;
#pragma unroll
    for (int j = 0; j < TK; ++j) {
      const int k = g + j * G;
      tdst[j] = k < n0 ? (T.segs[0][0] >> 1) + k : (k < n0 + n1 ? (T.segs[1][0] >> 1) + k - n0 : -1);
    }
  }
  const int num_actions = T.scheme == 1 ? 8 : 5;
  const bool keep = (flags & CZ_STEP_KEEP_ALL) != 0;
  const size_t na_stride = keep ? N * NA : 0;  // reward / flags of consecutive steps
  const int n2 = T.ranges[0][1] >> 1, o2 = T.ranges[0][0] >> 1, s2 = (T.ranges[0][0] - T.stage_lo) >> 1;
  const double2* tab_lane = reinterpret_cast<const double2*>(T.obs_table) + g;

  for (int k = 0; k < k_steps; ++k) {
    // ---- this step's actions: resident [K][n][A] array, or the counter stream of cz_random_actions
    uint32_t a_mine = 0;
    if (g < NA) {
      if (actions) {
        a_mine = a_next;  // requested one step ago: the load's latency hides behind a whole step
        if (k + 1 < k_steps) a_next = actions[((size_t)(k + 1) * N + env) * NA + g];
      } else {
        const double u = cz_uniform(seed ^ CZ_ACTION_STREAM, genv, 0, action_step + (uint64_t)k, (uint64_t)g);
        const int a = (int)(u * num_actions);
        a_mine = (uint32_t)(a < num_actions ? a : num_actions - 1);
      }
    }
    uint32_t act = 0;
#pragma unroll
    for (int i = 0; i < NA; ++i) act |= g_shfl(e, a_mine, i) << (8 * i);

    double rw[NA];
    uint32_t term_mask = 0, trunc_mask = 0;
    const bool fresh = (flags & CZ_STEP_AUTO_RESET) && (e.tinfo & TI_DONE);
    if (fresh) {
      // ---- CookingEnvironment.reset (cooking_env.py:178-210): pooled layout -> state, no step (cz_env_kernel)
      const int layout = cz_pick_layout(T.layout_cum, T.P, cz_mix(seed, genv, (uint64_t)e.episode));
      const uint32_t* src = T.pool + (size_t)layout * T.rows;
      e.rec = g < D ? __ldg(src + g) : 0u;
#pragma unroll
      for (int i = 0; i < NA; ++i) e.ag[i] = __ldg(src + D + i);
      e.sbits = __ldg(src + D + NA + CZ_ROW_SBITS);
      e.tinfo = __ldg(src + D + NA + CZ_ROW_TINFO);
      e.variant = __ldg(src + D + NA + CZ_ROW_VARIANT);
      e.episode += 1;
      wk_variant_consts(T, e);
    }
    wk_step_env(T, e, act, fresh, rw, term_mask, trunc_mask, seed, genv);
    if constexpr (STATS) {
      double r_mine[1] = {rw[0]};
#pragma unroll
      for (int i = 1; i < NA; ++i)
        if (g == i) r_mine[0] = rw[i];
      uint32_t served = 0, success = 0;
      if (cz_stats_rule<1>(st_seen, st_open, st_ret, r_mine, e.episode, e.tinfo, e.marks, T.R, T.end_all != 0, served, success)) {
        st_n += 1;
        st_len += TI_T(e.tinfo);
        st_served += served;
        st_succ += success;
        st_last = TI_T(e.tinfo) | served << 20 | success << 28;  // t < 2^20
        st_sum += st_ret[0];
        st_lret = st_ret[0];
      }
    }
    if (g < NA) {
      double r = rw[0];
#pragma unroll
      for (int i = 1; i < NA; ++i)
        if (g == i) r = rw[i];
      const size_t o = (size_t)k * na_stride + (size_t)env * NA + g;
      reward[o] = r;
      term[o] = (uint8_t)(term_mask >> g & 1u);
      trunc[o] = (uint8_t)(trunc_mask >> g & 1u);
    }

    // ---- get_feature_vector (cooking_env.py:352-373): the A rows of this step
    if (obs) {
      double2* g2 = reinterpret_cast<double2*>(obs + ((keep ? (size_t)k * N : 0) + (size_t)env) * NA * T.L);
#if CZ_WARP_TMA || CZ_WARP_WHOLE
      if (g == 0) cz_bulk_wait_read<0>();  // the TMA engine has read the staging rows of the previous step
#endif
      g_sync(e);  // the copy-out of the previous step has read the staging rows
      const double2* tab = tab_lane + (size_t)e.variant * 64 * tab2;
#if CZ_WARP_WHOLE
      // whole rows staged: the table segments of the NA rows go global -> their place in the rows (cp.async, no registers,
      // in flight under the pair stores), then ONE bulk store of the environment's NA * L doubles
#pragma unroll
      for (int a = 0; a < NA; ++a) {
        const double2* src = tab + A_XY(e.ag[a]) * tab2;
#pragma unroll
        for (int j = 0; j < TK; ++j)
          if (tdst[j] >= 0) cz_cp_async16(stage + a * stage2 + tdst[j], src + j * G);
      }
#endif
      for (int q0 = 0; q0 < n_pairs; q0 += G) {
        const int q = q0 + g;
        const bool live = q < n_pairs;
        wk_pair_store(T, e, live ? pmap[q] : 0u, live, sxl, syl, stage, stage2, CZ_WARP_WHOLE ? 0 : T.stage_lo);
      }
#if CZ_WARP_WHOLE
      cz_cp_async_wait_all();
      cz_fence_async_smem();  // generic-proxy and cp.async writes -> visible to the async proxy
      g_sync(e);
      if (g == 0) {
        cz_bulk_store_nocommit(g2, stage, (uint32_t)(NA * T.L) * 8u);
        cz_bulk_commit();
      }
#else
#if CZ_WARP_TMA
      // the computed range of the NA rows leaves through the TMA engine: one elected lane, one bulk store per row
      cz_fence_async_smem();  // generic-proxy writes -> visible to the async proxy
      g_sync(e);
      if (g == 0) {
#pragma unroll
        for (int a = 0; a < NA; ++a) cz_bulk_store_nocommit(g2 + a * L2 + o2, stage + a * stage2 + s2, (uint32_t)n2 * 16u);
        cz_bulk_commit();
      }
#else
      g_sync(e);
#pragma unroll
      for (int a = 0; a < NA; ++a)
        for (int q = g; q < n2; q += G) g2[a * L2 + o2 + q] = stage[a * stage2 + s2 + q];
#endif
#pragma unroll
      for (int a = 0; a < NA; ++a) {  // table segments of row a: loads first, then the stores
        const double2* src = tab + A_XY(e.ag[a]) * tab2;
        double2 v[TK];
#pragma unroll
        for (int j = 0; j < TK; ++j)
          if (tdst[j] >= 0) v[j] = __ldg(src + j * G);
#pragma unroll
        for (int j = 0; j < TK; ++j)
          if (tdst[j] >= 0) g2[a * L2 + tdst[j]] = v[j];
      }
#endif
    }
  }

#if CZ_WARP_TMA || CZ_WARP_WHOLE
  if (obs && g == 0) cz_bulk_wait_read<0>();  // the staging rows must outlive the last bulk stores
#endif
  // ---- registers -> state
  if (g < D) state[(size_t)g * N + env] = e.rec;
  if (g < NA + CZ_NUM_MISC_ROWS) {
    uint32_t w = wk_sel(e.ag, g);
    const int m = g - NA;
    if (m == CZ_ROW_SBITS) w = e.sbits;
    if (m == CZ_ROW_TINFO) w = e.tinfo;
    if (m == CZ_ROW_MARKS) w = e.marks;
    if (m == CZ_ROW_VARIANT) w = e.variant;
    if (m == CZ_ROW_RECIPES) w = e.rids;
    if (m == CZ_ROW_EPISODE) w = e.episode;
    state[(size_t)(D + g) * N + env] = w;
  }
  if (errflags && e.err && g == 0) errflags[env] |= e.err;
  if constexpr (STATS) {
    if (g < NA) S.ret[(size_t)env * NA + g] = st_ret[0];
    if (g == 0) {
      S.episode[env] = st_seen;
      S.open[env] = (uint8_t)st_open;
    }
    if (st_n) {  // at most one atomicAdd per field and environment per launch, whatever K is
      if (g < NA) {
        S.last_ret[(size_t)env * NA + g] = st_lret;
        atomicAdd(S.totals + 4 + g, st_sum);
      }
      if (g == 0) {
        S.last_len[env] = (int32_t)(st_last & 0xFFFFFu);
        S.last_served[env] = (uint8_t)((st_last >> 20) & 255u);
        S.last_success[env] = (uint8_t)(st_last >> 28);
        S.finished[env] += (int32_t)st_n;
        atomicAdd(S.totals + 0, (double)st_n);
        atomicAdd(S.totals + 1, (double)st_len);
        if (st_served) atomicAdd(S.totals + 2, (double)st_served);
        if (st_succ) atomicAdd(S.totals + 3, (double)st_succ);
      }
    }
  }
}
