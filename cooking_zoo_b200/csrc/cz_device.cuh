// cz_device.cuh — device-side data model and per-environment dynamics (sm_100a).
//
// One LANE owns one environment during the dynamics phase (scalar, table-driven code over a
// shared-memory column of packed object records); the WARP then cooperates on the
// observation rows of its 32 environments.  Citations: /root/reference/cooking_zoo/...
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/cz_b200.h"

// ---- device copy of the compiled tables (passed to kernels by value) ------------------
struct CzDev {
  int W, H, A, R, D, S, T, L, V, P, B, max_steps, end_all, grace, n_switches, n_blocks, rows;
  int scheme;  // 1 or 3: ActionScheme1 / ActionScheme3 (cooking_world/actions.py:2-17, 39-50)
  int n_comp, n_segs, n_ranges, tab_len;
  int segs[2][3];    // table segments of a row: {row offset, length, table offset} (doubles, even)
  int ranges[3][2];  // computed ranges of a row: {row offset, length}
  int stage_lo, stage_len;  // span of the computed ranges (what the staging buffer holds)
  // per-lane constants of the packed (observer, slot) layout, filled by cz_tables_create
  const int4* lane_map;  // [32] {computed-slot descriptor or -1, observer, t0, t1}: global memory (dynamic indexing of kernel
                         // parameters would force a local-memory copy of the whole struct)
  double r_node, r_recipe, r_penalty, r_time, respawn, despawn;
  const double* xlut;
  const double* ylut;
  const uint8_t* grid;
  const uint8_t* static_cells;
  const uint8_t* scan_order;
  const uint8_t* special_cells;
  const uint64_t* static_masks;
  const uint8_t* slot_type;
  const uint8_t* type_flags;
  const uint8_t* type_base;
  const uint8_t* type_count;
  const uint32_t* comp_slots;
  const double* obs_table;
  const uint32_t* recipe_nodes;
  const uint32_t* recipe_spans;  // [B][8] per node: first slot | slots << 8 | required record bits << 16 (cz_tables_create)
  const uint8_t* recipe_len;
  const uint32_t* pool;
  const uint8_t* default_recipes;
  const uint8_t* spawn_x;
  const uint8_t* spawn_y;
  const uint8_t* spawn_n;
  const float* xlut32;       // the same tables rounded to float32 once on the host (float32 observation rows)
  const float* ylut32;
  const float* obs_table32;
  const uint64_t* layout_cum;  // weighted layout pool: cumulative probabilities * 2^64, or nullptr (uniform pool)
  const void* blob;  // BlockSmem image (LUTs + SmemTabs), built by cz_tables_create
};

// Small lookup tables staged in shared memory by every block (with 214 KB of shared memory in
// use the L1 is only ~14 KB, so a __ldg of these is an L2 round trip in the middle of a
// dependent chain).  Kernels instantiated with FAST=true require V <= CZ_SV and B <= CZ_SB and
// read the shared copy; FAST=false reads global memory.
#define CZ_SV 16
#define CZ_SB 16
struct VarTabs {  // per static variant (272 B); only the V variants of the tables occupy shared memory
  uint64_t static_masks[8];
  uint8_t grid[64];
  uint8_t scan_order[CZ_MAX_DYN];
  uint8_t special_cells[4 * CZ_MAX_SPECIAL];
  uint8_t static_cells[CZ_MAX_STATIC_SLOTS];
};
struct SmemTabs {
  uint32_t recipe_nodes[CZ_SB][CZ_MAX_NODES];
  uint32_t recipe_spans[CZ_SB][CZ_MAX_NODES];
  uint8_t slot_tf[CZ_MAX_DYN];  // type_flags[slot_type[s]]
  uint8_t slot_type[CZ_MAX_DYN];
  uint8_t type_base[CZ_MAX_TYPES];
  uint8_t type_count[CZ_MAX_TYPES];
  uint8_t recipe_len[CZ_SB];
  uint8_t recipe_desc[CZ_SB][CZ_MAX_NODES];  // per node: bit j set iff node j is the node itself or one of its descendants (cz_warp.cuh)
  VarTabs var[1];  // [V], V <= CZ_SV
};

// static kinds (grid low nibble) — cooking_zoo_b200/entities.py ST_*
enum { ST_NONE = 0, ST_FLOOR, ST_COUNTER, ST_CUTBOARD, ST_BLENDER, ST_DELIVER, ST_SWITCH, ST_BLOCK };
// dynamic type flags
enum { TF_PLATE = 1, TF_CHOP = 2, TF_BLEND = 4, TF_SPAWN = 8 };
// feature layouts
enum { FV_NONE = 0, FV_ONE, FV_CHOP, FV_CHOPBLEND, FV_AGENT, FV_SWITCH, FV_BLOCK };

// ---- packed records (cz_b200.h) ----------------------------------------------------------
#define O_XY(r) ((r) & 63u)
#define O_PRESENT 64u
#define O_CHOP 128u
#define O_MASH 256u
#define O_FREE 512u
#define O_CK(r) (((r) >> 10) & 3u)
#define O_CID(r) (((r) >> 12) & 31u)
#define O_POS(r) (((r) >> 17) & 63u)
#define O_PCOUNT(r) (((r) >> 23) & 127u) /* Plate records: items on the plate (kept by the merge / pick-up-special paths) */
#define O_PCOUNT_ONE (1u << 23)
#define O_WITH_XY(r, xy) (((r) & ~63u) | (xy))
#define O_WITH_CONT(r, k, id, pos) (((r) & 0xFF8003FFu) | ((uint32_t)(k) << 10) | ((uint32_t)(id) << 12) | ((uint32_t)(pos) << 17))
// one masked compare instead of three field tests (hot inner loops of the dynamics)
#define O_AT(r, cell) (((r) & 0x7Fu) == ((cell) | O_PRESENT))                             /* present, at cell */
#define O_IN_STATIC_AT(r, cell) (((r) & 0xC7Fu) == ((cell) | O_PRESENT | (1u << 10)))      /* ... as content of the static object */
#define O_ON_PLATE(r, p) (((r) & 0x1FC40u) == (O_PRESENT | (2u << 10) | ((uint32_t)(p) << 12))) /* present, content of plate p */
#define CK_HELD 0u
#define CK_STATIC 1u
#define CK_PLATE 2u

#define A_XY(r) ((r) & 63u)
#define A_ORI(r) (((r) >> 6) & 7u)
#define A_HAS(r) (((r) >> 9) & 1u)
#define A_HOLD(r) (((r) >> 10) & 31u)
#define A_ACTIVE(r) (((r) >> 15) & 1u)
#define A_GRACE(r) ((r) >> 16)

#define SB_CUT_READY(k) (1u << (k))
#define SB_BL_READY(k) (1u << (4 + (k)))
#define SB_BL_TOGGLE(k) (1u << (8 + (k)))
#define SB_SW_ACTIVE(k) (1u << (12 + (k)))
#define SB_BLK_WALK(k) (1u << (16 + (k)))

#define TI_T(x) ((x) & 0xFFFFFu)
#define TI_DONE (1u << 20)
#define TI_NLIVE(x) (((x) >> 21) & 7u)

#define TAB_GRID(v, c) (FAST ? (uint32_t)st->var[v].grid[c] : (uint32_t)__ldg(T.grid + (v) * 64 + (c)))
#define TAB_SCAN(v, k) (FAST ? (uint32_t)st->var[v].scan_order[k] : (uint32_t)__ldg(T.scan_order + (v) * T.D + (k)))
#define TAB_SPECIAL(v, kind, k) \
  (FAST ? (uint32_t)st->var[v].special_cells[(kind) * CZ_MAX_SPECIAL + (k)] \
               : (uint32_t)__ldg(T.special_cells + ((v) * 4 + (kind)) * CZ_MAX_SPECIAL + (k)))
#define TAB_SCELL(v, i) (FAST ? (uint32_t)st->var[v].static_cells[i] : (uint32_t)__ldg(T.static_cells + (v) * T.S + (i)))
#define TAB_SMASK(v, k) (FAST ? st->var[v].static_masks[k] : __ldg(T.static_masks + (v) * 8 + (k)))
#define TAB_RNODE(b, k) (FAST ? st->recipe_nodes[b][k] : __ldg(T.recipe_nodes + (b) * CZ_MAX_NODES + (k)))
#define TAB_RSPAN(b, k) (FAST ? st->recipe_spans[b][k] : __ldg(T.recipe_spans + (b) * CZ_MAX_NODES + (k)))
#define TAB_RLEN(b) (FAST ? (uint32_t)st->recipe_len[b] : (uint32_t)__ldg(T.recipe_len + (b)))
#define TAB_TF(s) (FAST ? (uint32_t)st->slot_tf[s] : (uint32_t)__ldg(T.type_flags + __ldg(T.slot_type + (s))))
#define TAB_STYPE(s) (FAST ? (uint32_t)st->slot_type[s] : (uint32_t)__ldg(T.slot_type + (s)))
#define TAB_TBASE(t) (FAST ? (int)st->type_base[t] : (int)__ldg(T.type_base + (t)))
#define TAB_TCOUNT(t) (FAST ? (int)st->type_count[t] : (int)__ldg(T.type_count + (t)))

#define OSTRIDE 33  // shared-memory column stride (words): lane-per-env and lane-per-slot are both conflict-free

// Per-lane view of one environment.  Object records live in a shared-memory column.
struct EnvRegs {
  uint32_t* o;   // &sobj[lane]; dynamic slot s at o[s * OSTRIDE]
  uint32_t* ag;  // &sag[lane];  agent i at ag[i * OSTRIDE]
  const SmemTabs* st;
  uint32_t sbits, tinfo, marks, variant, rids, episode, err;
};

__device__ __forceinline__ uint64_t cz_mix(uint64_t seed, uint64_t env, uint64_t episode) {
  // splitmix64 finaliser over a counter built from (seed, env, episode)
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (env + 1) + 0xD1B54A32D192ED03ull * (episode + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// Pool index selected by a 64-bit draw: first layout whose cumulative threshold exceeds it (weighted pool: the exact
// distribution of the reference's level parser), or draw % P (uniform pool).  Host twin: cz_layout_index.
__host__ __device__ __forceinline__ int cz_pick_layout(const uint64_t* cum, int P, uint64_t u) {
  if (!cum) return (int)(u % (uint64_t)P);
  int lo = 0, hi = P - 1;  // cum[P - 1] = 2^64 - 1 >= u: the answer exists
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
#ifdef __CUDA_ARCH__
    const uint64_t c = __ldg(cum + mid);
#else
    const uint64_t c = cum[mid];
#endif
    if (c > u) hi = mid; else lo = mid + 1;
  }
  return lo;
}

template <bool FAST>
__device__ __forceinline__ bool cz_walkable(const CzDev& T, const EnvRegs& e, uint32_t cell) {
  // StaticObject.walkable (world_objects.py:20,148,199): Floor and Switch always, Block by state
  const SmemTabs* st = e.st;
  uint32_t g = TAB_GRID(e.variant, cell);
  uint32_t kind = g & 15u;
  if (kind == ST_FLOOR || kind == ST_SWITCH) return true;
  if (kind == ST_BLOCK) return (e.sbits & SB_BLK_WALK(g >> 4)) != 0;
  return false;
}

// c-th uniform draw of environment `env` in step `t` of episode `episode` (cz_spawn_uniform)
__host__ __device__ __forceinline__ double cz_uniform(uint64_t seed, uint64_t env, uint64_t episode, uint64_t t, uint64_t c) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (env + 1) + 0xD1B54A32D192ED03ull * (episode + 1) +
               0x8CB92BA72F3D8DD7ull * (t + 1) + 0xF1357AEA2E62A9C5ull * (c + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ bool cz_agent_on(const CzDev& T, const EnvRegs& e, uint32_t cell) {
  // `any(agent.location == interaction_location for agent in self.agents)` (cooking_world.py:116,158)
  bool on = false;
#pragma unroll 1
  for (int j = 0; j < T.A; ++j)
    if (A_XY(e.ag[j * OSTRIDE]) == cell) on = true;
  return on;
}

// Move a dynamic object (and, for a Plate, its content) — Object.move_to / Plate.move_to
// (abstract_classes.py:21-22, world_objects.py:393-396).
template <bool FAST>
__device__ __forceinline__ void cz_move_obj(const CzDev& T, EnvRegs& e, uint32_t s, uint32_t xy) {
  const uint32_t rec = e.o[s * OSTRIDE];
  e.o[s * OSTRIDE] = O_WITH_XY(rec, xy);
  const SmemTabs* st = e.st;
  if ((TAB_TF(s) & TF_PLATE) && O_PCOUNT(rec)) {  // an empty plate (the common case) has nothing to carry along
    #pragma unroll 1
    for (int k = 0; k < T.D; ++k) {
      uint32_t r = e.o[k * OSTRIDE];
      if (O_ON_PLATE(r, s)) e.o[k * OSTRIDE] = O_WITH_XY(r, xy);
    }
  }
}

// list.remove(obj) on the content of the static object at `cell`: later items shift down.
__device__ __forceinline__ void cz_remove_from_static(const CzDev& T, EnvRegs& e, uint32_t cell, uint32_t pos) {
  #pragma unroll 1
  for (int k = 0; k < T.D; ++k) {
    uint32_t r = e.o[k * OSTRIDE];
    if (O_IN_STATIC_AT(r, cell) && O_POS(r) > pos) e.o[k * OSTRIDE] = r - (1u << 17);
  }
}

// add_content's `for c in content: c.free = False; content[-1].free = True` for a plate
// (world_objects.py:398-406): clear the flag of everything already on plate `p`.
__device__ __forceinline__ void cz_plate_clear_free(const CzDev& T, EnvRegs& e, uint32_t p) {
  #pragma unroll 1
  for (int k = 0; k < T.D; ++k) {
    uint32_t r = e.o[k * OSTRIDE];
    if (O_ON_PLATE(r, p)) e.o[k * OSTRIDE] = r & ~O_FREE;
  }
}

// resolve_interaction -> resolve_execute_action | resolve_primary_interaction -> attempt_merge
// (action_scheme3.py:37-43, cooking_world.py:114-136, 156-170, 243-261).
// mode: 0 = scheme3 (execute iff an action object holds something unfinished, else primary),
//       5 / 6 / 7 = scheme1's INTERACT_PRIMARY / INTERACT_PICK_UP_SPECIAL / EXECUTE_ACTION (action_scheme1.py:33-40).
// Returns the plate whose content lost an item (its free flags are refreshed at the end of the step) or 0xFF.
// `stale` is set when the static container at `cell` keeps items whose free flags must be refreshed in
// progress_world (it lost one of several items, or a chopped Bread spawned its twin on top).
template <bool FAST>
__device__ __forceinline__ uint32_t cz_interact(const CzDev& T, EnvRegs& e, int i, uint32_t cell, uint32_t mode, bool& stale) {
  const uint32_t agent_rec = e.ag[i * OSTRIDE];
  const SmemTabs* st = e.st;
  const uint32_t g = TAB_GRID(e.variant, cell);
  const uint32_t kind = g & 15u, sp = g >> 4;
  // one pass in scan order over the dynamic objects at the faced cell (cooking_world.py:232-241)
  int n_dyn = 0, last = -1, first_free = -1, n_plates = 0, plate = -1, n_content = 0;
  bool any_not_done = false;
  for (int k = 0; k < T.D; ++k) {
    int s = TAB_SCAN(e.variant, k);
    uint32_t r = e.o[s * OSTRIDE];
    if (!O_AT(r, cell)) continue;
    ++n_dyn;
    last = s;
    if (first_free < 0 && (r & O_FREE)) first_free = s;
    if (TAB_TF(s) & TF_PLATE) {
      ++n_plates;
      plate = s;
    } else if (!(r & (O_CHOP | O_MASH))) {
      any_not_done = true;  // Food.done() (world_objects.py:441,549,...)
    }
    if (O_CK(r) == CK_STATIC) ++n_content;
  }
  const bool blocked = cz_agent_on(T, e, cell);

  if (mode == 6u) {
    // ---- resolve_interaction_pick_up_special (cooking_world.py:138-154): take the last item off the one plate
    if (blocked || A_HAS(agent_rec) || n_dyn == 0 || n_plates != 1) return 0xFFu;
    int top = -1, ts = -1;
    #pragma unroll 1
    for (int k = 0; k < T.D; ++k) {
      uint32_t r = e.o[k * OSTRIDE];
      if (O_ON_PLATE(r, plate) && (int)O_POS(r) > top) { top = O_POS(r); ts = k; }
    }
    if (ts < 0) return 0xFFu;  // content.pop(-1) on an empty plate: IndexError, swallowed
    e.o[plate * OSTRIDE] -= O_PCOUNT_ONE;
    e.o[ts * OSTRIDE] = O_WITH_XY(O_WITH_CONT(e.o[ts * OSTRIDE], CK_HELD, i, 0), A_XY(agent_rec));
    e.ag[i * OSTRIDE] = (agent_rec & ~(0x3Fu << 9)) | (1u << 9) | ((uint32_t)ts << 10);
    return (uint32_t)plate;
  }
  if (mode == 7u || (mode == 0u && (kind == ST_CUTBOARD || kind == ST_BLENDER) && any_not_done)) {
    // ---- resolve_execute_action (cooking_world.py:156-170)
    if (blocked) return 0xFFu;
    if (kind != ST_CUTBOARD && kind != ST_BLENDER) return 0xFFu;  // not an ActionObject
    if (kind == ST_CUTBOARD) {  // Cutboard.action (world_objects.py:250-269)
      if (!(e.sbits & SB_CUT_READY(sp))) return 0xFFu;
      for (int p = 0; p < n_content; ++p) {
        int s = -1;
        #pragma unroll 1
        for (int k = 0; k < T.D; ++k) {
          uint32_t r = e.o[k * OSTRIDE];
          if (O_IN_STATIC_AT(r, cell) && O_POS(r) == (uint32_t)p) s = k;
        }
        if (s < 0) break;
        uint32_t r = e.o[s * OSTRIDE];
        uint32_t tid = TAB_STYPE(s);
        uint32_t tf = TAB_TF(s);
        if (!(tf & TF_CHOP)) return 0xFFu;
        if (r & O_CHOP) continue;  // ChopFood.chop / Bread.chop: already chopped -> not executed
        e.o[s * OSTRIDE] = r | O_CHOP;
        e.sbits &= ~SB_CUT_READY(sp);
        if (tf & TF_SPAWN) {  // Bread.chop spawns a chopped twin (world_objects.py:738-745)
          int base = TAB_TBASE(tid), cnt = TAB_TCOUNT(tid);
          int slot = -1;
          #pragma unroll 1
          for (int k = base; k < base + cnt; ++k)
            if (slot < 0 && !(e.o[k * OSTRIDE] & O_PRESENT)) slot = k;
          if (slot < 0) {
            e.err |= CZ_ERR_OBS_OVERFLOW;  // the reference's obs vector would grow (cooking_env.py:371)
          } else {
            e.o[slot * OSTRIDE] = O_WITH_CONT(cell | O_PRESENT | O_CHOP | O_FREE, CK_STATIC, 0, n_content);
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
    if (kind == ST_DELIVER) rel = false;  // world_objects.py:117-118
    else if (kind == ST_CUTBOARD) {  // :275-278
      if (n_content == 1) e.sbits &= ~SB_CUT_READY(sp);
    } else if (kind == ST_BLENDER) {  // :340-346
      if (e.sbits & SB_BL_TOGGLE(sp)) rel = false;
      else if (n_content - 1 == 0) e.sbits &= ~SB_BL_READY(sp);
    }
    if (!rel) return 0xFFu;
    int gs = first_free >= 0 ? first_free : last;
    uint32_t r = e.o[gs * OSTRIDE];
    if (O_CK(r) != CK_STATIC) return 0xFFu;  // `object_to_grab in static_object.content`
    if (n_content > 1) {  // a lone item leaves nothing behind to shift or to refresh
      cz_remove_from_static(T, e, cell, O_POS(r));
      stale = true;
    }
    e.o[gs * OSTRIDE] = O_WITH_CONT(r, CK_HELD, i, 0);
    cz_move_obj<FAST>(T, e, gs, axy);  // Agent.grab (world_objects.py:786-788)
    e.ag[i * OSTRIDE] = (agent_rec & ~(0x3Fu << 9)) | (1u << 9) | ((uint32_t)gs << 10);
    return 0xFFu;
  }

  // ---- attempt_merge (cooking_world.py:243-261)
  const uint32_t h = A_HOLD(agent_rec);
  const uint32_t hr = e.o[h * OSTRIDE];
  const uint32_t htf = TAB_TF(h);
  const uint32_t dropped = agent_rec & ~(0x3Fu << 9);
  if (n_plates == 1) {
    // Plate.accepts: Food and done and room (world_objects.py:408-409)
    if ((htf & (TF_CHOP | TF_BLEND)) && (hr & (O_CHOP | O_MASH))) {
      const uint32_t n = O_PCOUNT(e.o[plate * OSTRIDE]);
      if (n < 64) {
        if (n) cz_plate_clear_free(T, e, plate);
        e.o[plate * OSTRIDE] += O_PCOUNT_ONE;
        e.o[h * OSTRIDE] = O_WITH_XY(O_WITH_CONT(hr, CK_PLATE, plate, n) | O_FREE, cell);
        e.ag[i * OSTRIDE] = dropped;  // put_down (world_objects.py:790-792)
      }
    }
  } else if ((htf & TF_PLATE) && n_dyn > 0) {
    uint32_t pr = e.o[last * OSTRIDE];
    uint32_t ptf = TAB_TF(last);
    if ((ptf & (TF_CHOP | TF_BLEND)) && (pr & (O_CHOP | O_MASH))) {
      const uint32_t n = O_PCOUNT(hr);
      if (n < 64) {
        if (n) cz_plate_clear_free(T, e, h);
        e.o[h * OSTRIDE] = hr + O_PCOUNT_ONE;
        if (O_CK(pr) == CK_STATIC) {
          if (n_content > 1) {
            cz_remove_from_static(T, e, cell, O_POS(pr));
            stale = true;
          }
        } else {
          e.err |= CZ_ERR_REMOVE;
        }
        e.o[last * OSTRIDE] = O_WITH_XY(O_WITH_CONT(pr, CK_PLATE, h, n) | O_FREE, axy);
      }
    }
  } else {
    bool ok = false;  // StaticObject.accepts
    if (kind == ST_COUNTER || kind == ST_DELIVER) ok = n_content < 1;  // :64-66, :107-108
    else if (kind == ST_CUTBOARD) ok = (htf & TF_CHOP) && n_content < 1 && !(hr & O_CHOP);  // :271-273
    else if (kind == ST_BLENDER)
      ok = (htf & TF_BLEND) && !(e.sbits & SB_BL_TOGGLE(sp)) && n_content + 1 <= 1 && !(hr & O_MASH);  // :337-338
    if (ok) {
      if (kind == ST_CUTBOARD) e.sbits |= SB_CUT_READY(sp);
      if (kind == ST_BLENDER) e.sbits |= SB_BL_READY(sp);
      e.o[h * OSTRIDE] = O_WITH_CONT(hr, CK_STATIC, 0, n_content) | O_FREE;
      cz_move_obj<FAST>(T, e, h, cell);
      e.ag[i * OSTRIDE] = dropped;
    }
  }
  return 0xFFu;
}

// progress_world's free-flag refresh for one static container (cooking_world.py:82-88):
// only containers that lost an item or gained a spawned Bread this step can be stale.
__device__ __forceinline__ void cz_refresh_static_free(const CzDev& T, EnvRegs& e, uint32_t cell) {
  int top = -1;
  #pragma unroll 1
  for (int k = 0; k < T.D; ++k) {
    uint32_t r = e.o[k * OSTRIDE];
    if (O_IN_STATIC_AT(r, cell) && (int)O_POS(r) > top) top = O_POS(r);
  }
  #pragma unroll 1
  for (int k = 0; k < T.D; ++k) {
    uint32_t r = e.o[k * OSTRIDE];
    if (O_IN_STATIC_AT(r, cell))
      e.o[k * OSTRIDE] = ((int)O_POS(r) == top) ? (r | O_FREE) : (r & ~O_FREE);
  }
}

// The same for a plate that lost its top item (scheme1's pick-up-special).
__device__ __forceinline__ void cz_refresh_plate_free(const CzDev& T, EnvRegs& e, uint32_t p) {
  int top = -1;
  #pragma unroll 1
  for (int k = 0; k < T.D; ++k) {
    uint32_t r = e.o[k * OSTRIDE];
    if (O_ON_PLATE(r, p) && (int)O_POS(r) > top) top = O_POS(r);
  }
  #pragma unroll 1
  for (int k = 0; k < T.D; ++k) {
    uint32_t r = e.o[k * OSTRIDE];
    if (O_ON_PLATE(r, p))
      e.o[k * OSTRIDE] = ((int)O_POS(r) == top) ? (r | O_FREE) : (r & ~O_FREE);
  }
}

// Cells holding an object that satisfies one recipe node on its own (type + condition):
// the `for obj in world.world_objects[node.name]` loop of Recipe.update_recipe_state
// (recipe.py:83-87) with check_conditions' attribute test (:96-98).  Out of line: it is called
// for every node of every recipe and would otherwise be replicated by the unrolled caller.
template <int S = OSTRIDE>  // S: words between slot records (1: the warp kernel's cook scratch, cz_policy_dev.cuh)
__device__ __noinline__ uint64_t cz_node_mask(const uint32_t* o, uint32_t span) {
  const uint32_t need = span >> 16;  // O_PRESENT plus the chopped / mashed bit the node asks for
  const int base = span & 255u, end = base + ((span >> 8) & 255u);  // no slots: a type the meta file does not know
  uint64_t mask = 0;
  for (int s = base; s < end; ++s) {
    uint32_t r = o[s * S];
    if ((r & need) == need) mask |= 1ull << O_XY(r);
  }
  return mask;
}

// Recipe.update_recipe_state as cell bitmasks (recipe.py:77-104): node mask = cells holding an
// object of the node's type that meets its condition, ANDed with every child's mask (children
// come later in node_list, so the list is walked back to front).
// Out of line and by value (the environment view stays in registers): one copy of the unrolled node walk serves the
// step, the auto-reset and the reset kernels; the dynamics are instruction-fetch bound, code size is the budget.
template <bool FAST>
__device__ __noinline__ uint32_t cz_recipe_marks_of(const CzDev& T, const uint32_t* eo, const SmemTabs* st, uint32_t variant,
                                                    uint32_t rid) {
  struct { const uint32_t* o; uint32_t variant; } e = {eo, variant};
  uint64_t m[CZ_MAX_NODES];
  const int n = TAB_RLEN(rid);
  uint32_t marks = 0;
#pragma unroll
  for (int k = CZ_MAX_NODES - 1; k >= 0; --k) {
    m[k] = 0;
    if (k < n) {
      const uint32_t node = TAB_RNODE(rid, k);
      const uint32_t kids = node >> 16;
      uint64_t mask = ~0ull;
      if (kids) {  // leaves (most nodes) skip the child loop
#pragma unroll
        for (int j = k + 1; j < CZ_MAX_NODES; ++j)
          if (kids & (1u << j)) mask &= m[j];
      }
      // a node whose children are not all satisfied at some common cell cannot be marked whatever lies on its own
      // cells: its slots are only looked at when the children leave a candidate cell (most steps: none)
      if (mask) mask &= (node & 256u) ? TAB_SMASK(e.variant, node & 7u) : cz_node_mask(e.o, TAB_RSPAN(rid, k));
      m[k] = mask;
      if (mask) marks |= 1u << k;
    }
  }
  return marks;
}
template <bool FAST>
__device__ __forceinline__ uint32_t cz_recipe_marks(const CzDev& T, const EnvRegs& e, uint32_t rid) {
  return cz_recipe_marks_of<FAST>(T, e.o, e.st, e.variant, rid);
}

// CookingEnvironment.accumulated_step (cooking_env.py:243-269) for one environment.
// Writes reward f64[A], terminated u8[A], truncated u8[A] of this environment.
template <bool FAST, int NA>
__device__ __forceinline__ void cz_step_env(const CzDev& T, EnvRegs& e, const uint32_t act_packed,
                                            double* __restrict__ reward, uint8_t* __restrict__ term_out,
                                            uint8_t* __restrict__ trunc_out, uint64_t seed, uint64_t genv) {
  const int A = NA ? NA : T.A;  // compile-time agent count in the specialised kernels
  const bool scheme1 = T.scheme == 1;
  const SmemTabs* st = e.st;
  const uint32_t t = TI_T(e.tinfo) + 1;  // :244
  uint32_t active = 0;
  for (int i = 0; i < A; ++i)
    if (A_ACTIVE(e.ag[i * OSTRIDE])) active |= 1u << i;
  uint32_t changed = 0;

  // ---- action_scheme3.perform_agent_actions (action_scheme3.py:4-16)
  // per agent, 8 bits each: apack = action after checks, fpack = faced cell, epack = end cell | 0x40 walkable
  uint32_t apack = 0, fpack = 0, epack = 0x80808080u;
#pragma unroll 1
  for (int i = 0; i < A; ++i) {
    if (!(active >> i & 1u)) continue;
    uint32_t ai = (act_packed >> (8 * i)) & 255u;
    if (ai > (scheme1 ? 7u : 4u)) ai = 0;  // outside the action space: behaves as a no-op
    uint32_t rec = e.ag[i * OSTRIDE];
    int x = rec & 7u, y = (rec >> 3) & 7u;
    uint32_t faced = A_XY(rec);
    if (ai >= 1u && ai <= 4u) {
      rec = (rec & ~(7u << 6)) | (ai << 6);  // change_orientation even if cancelled later (:8-10)
      e.ag[i * OSTRIDE] = rec;
      int tx = x + (ai == 2) - (ai == 1), ty = y + (ai == 3) - (ai == 4);  // cooking_world.py:172-184
      if (tx < 0 || ty < 0 || tx > T.W - 1 || ty > T.H - 1) ai = 0;  // check_inbounds :192-204
      else faced = (uint32_t)(tx | ty << 3);
    }
    // check_collisions, first loop (:206-216); scheme1's interact actions target the agent's own cell
    uint32_t tgt = (ai >= 1u && ai <= 4u) ? faced : A_XY(rec);
    bool w = cz_walkable<FAST>(T, e, tgt);
    uint32_t endc = (w ? tgt : A_XY(rec)) | (w ? 0x40u : 0u);
    apack |= ai << (8 * i);
    fpack |= faced << (8 * i);
    epack = (epack & ~(0xFFu << (8 * i))) | (endc << (8 * i));
  }
  // check_collisions, second loop (:217-221): one pass over pre-move end cells
  uint32_t cancel = 0;
  for (int i = 0; i < A; ++i) {
    uint32_t ei = (epack >> (8 * i)) & 255u;
    if (!(ei & 0x40u) || (ei & 0x80u)) continue;  // not walkable, or inactive
    for (int j = 0; j < A; ++j) {
      uint32_t ej = (epack >> (8 * j)) & 255u;
      if (j != i && !(ej & 0x80u) && (ej & 63u) == (ei & 63u)) cancel |= 1u << i;
    }
  }
  // sequential resolution in agent order (action_scheme3.py:15-34).  The loop stays rolled and cz_interact has ONE
  // call site: the dynamics are bound by instruction fetch (profiles/r02_notes.md), so code size is the budget.
  uint32_t pressed = 0, dirty = 0xFFFFFFFFu, dirty_plate = 0xFFFFFFFFu;
#pragma unroll 1
  for (int i = 0; i < A; ++i) {
    if (!(active >> i & 1u)) continue;
    uint32_t rec = e.ag[i * OSTRIDE];
    const uint32_t ai = (cancel >> i & 1u) ? 0u : ((apack >> (8 * i)) & 255u);
    uint32_t cell = 0, mode = 0;
    bool interact = false;
    if (scheme1) {
      if (ai == 0u) continue;  // scheme1: only walk actions walk (action_scheme1.py:16-19), a no-op does nothing
      if (ai >= 5u) {          // interact with the cell the agent faces (cooking_world.py:115,139,157)
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
      if (cz_walkable<FAST>(T, e, tgt)) {  // resolve_walking_action (:26-34)
        rec = (rec & ~63u) | tgt;
        e.ag[i * OSTRIDE] = rec;
        if (A_HAS(rec)) cz_move_obj<FAST>(T, e, A_HOLD(rec), tgt);  // Agent.move_to (world_objects.py:793-796)
        uint32_t g = TAB_GRID(e.variant, tgt);
        if ((g & 15u) == ST_SWITCH) {  // Switch.add_content (:159-163)
          e.sbits ^= SB_SW_ACTIVE(g >> 4);
          pressed |= 1u << (g >> 4);
        }
      } else if (ai && !scheme1) {
        cell = tgt;
        interact = true;
      }
    }
    if (interact) {
      bool stale = false;
      const uint32_t p = cz_interact<FAST>(T, e, i, cell, mode, stale);  // p != 0xFF only for scheme1's pick-up-special
      if (stale) dirty = (dirty & ~(0xFFu << (8 * i))) | (cell << (8 * i));
      dirty_plate = (dirty_plate & ~(0xFFu << (8 * i))) | (p << (8 * i));
    }
  }

  // ---- progress_world (cooking_world.py:77-88)
  if (e.sbits & (0xFu << 8)) {  // some blender is switched on: Blender.process (world_objects.py:321-335)
    for (int k = 0; k < CZ_MAX_SPECIAL; ++k) {
      if (!(e.sbits & SB_BL_TOGGLE(k))) continue;
      uint32_t cell = TAB_SPECIAL(e.variant, 1, k);
      if (cell == 0xFFu) continue;
      int n = 0;
      bool all_mashed = true;
      #pragma unroll 1
      for (int s = 0; s < T.D; ++s) {
        uint32_t r = e.o[s * OSTRIDE];
        if (!O_IN_STATIC_AT(r, cell)) continue;
        ++n;
        if (!(r & (O_CHOP | O_MASH))) {  // BlenderFood.blend: one call takes FRESH to MASHED (abstract_classes.py:266-273)
          r |= O_MASH;
          e.o[s * OSTRIDE] = r;
        }
        if (!(r & O_MASH)) all_mashed = false;
      }
      if (n > 0 && all_mashed) e.sbits &= ~(SB_BL_TOGGLE(k) | SB_BL_READY(k));
    }
  }
  if (dirty != 0xFFFFFFFFu) {
    for (int i = 0; i < A; ++i) {
      uint32_t c = (dirty >> (8 * i)) & 255u;
      if (c != 0xFFu) cz_refresh_static_free(T, e, c);
    }
  }
  if (dirty_plate != 0xFFFFFFFFu) {
    for (int i = 0; i < A; ++i) {
      uint32_t p = (dirty_plate >> (8 * i)) & 255u;
      if (p != 0xFFu) cz_refresh_plate_free(T, e, p);
    }
  }
  // ---- resolve_linked_interactions (cooking_world.py:90-92; Switch :165-169, Block :215-216)
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
  // ---- handle_agent_spawn (cooking_world.py:267-277).  At the default rates 0.0 the reference's
  // draws change nothing, so only the grace countdown remains.
  if (T.respawn > 0.0 || T.despawn > 0.0) {
    uint32_t c = 0;  // draws consumed by this environment this step
    for (int i = 0; i < A; ++i) {
      uint32_t rec = e.ag[i * OSTRIDE];
      if (A_GRACE(rec) > 0) { e.ag[i * OSTRIDE] = rec - (1u << 16); continue; }
      const bool act_i = active >> i & 1u;
      if (__popc(active) > 1 && act_i) {  // short-circuit order of :273-274: the draw happens only here
        if (cz_uniform(seed, genv, e.episode, t, c++) < T.despawn) {
          if (!A_HAS(rec)) {  // despawn_agent :279-284: no-op while holding
            active &= ~(1u << i);
            changed |= 1u << i;
          }
        }
      } else if (!act_i) {
        if (cz_uniform(seed, genv, e.episode, t, c++) < T.respawn) {  // respawn_agent :286-290
          active |= 1u << i;
          changed |= 1u << i;
          const int nx = __ldg(T.spawn_n + 2 * i), ny = __ldg(T.spawn_n + 2 * i + 1);
          uint32_t cell = A_XY(rec);
          bool found = false;
          for (int tries = 0; tries < 1002 && !found; ++tries) {  // parsing.generate_location :154-167
            int x = __ldg(T.spawn_x + 8 * i + min(nx - 1, (int)(cz_uniform(seed, genv, e.episode, t, c++) * nx)));
            int y = __ldg(T.spawn_y + 8 * i + min(ny - 1, (int)(cz_uniform(seed, genv, e.episode, t, c++) * ny)));
            uint32_t cand = (uint32_t)(x | y << 3);
            if (x < T.W && y < T.H && (TAB_GRID(e.variant, cand) & 15u) == ST_FLOOR && !cz_agent_on(T, e, cand)) {
              cell = cand;
              found = true;
            }
          }
          if (!found) e.err |= CZ_ERR_SPAWN_LOC;
          e.ag[i * OSTRIDE] = (rec & 0xFFC0u) | cell | ((uint32_t)T.grace << 16);
        }
      }
    }
  } else {
    for (int i = 0; i < A; ++i)
      if (A_GRACE(e.ag[i * OSTRIDE]) > 0) e.ag[i * OSTRIDE] -= 1u << 16;
  }

  uint32_t relevant = active | changed;  // compute_relevant_agents :292

  // ---- compute_rewards / compute_truncated (cooking_env.py:290-350)
  const bool time_up = t >= (uint32_t)T.max_steps;
  uint32_t trunc_mask = 0;
  if (time_up) {
    if (TI_NLIVE(e.tinfo) < (uint32_t)A) e.err |= CZ_ERR_TRUNC_DESPAWN;
    trunc_mask = relevant;
    changed = relevant;
    active = 0;
  }
  trunc_mask |= changed & ~active & relevant;
  relevant = active | changed;
  // agent i is the k-th relevant agent and receives entry k of the recipe lists (:250-262)
  uint32_t new_marks = 0;
  bool all_done = true, any_done = false;
#pragma unroll 1
  for (int r = 0; r < T.R; ++r) {
    uint32_t rid = (e.rids >> (8 * r)) & 255u;
    uint32_t before = (e.marks >> (8 * r)) & 255u;
    uint32_t after = cz_recipe_marks<FAST>(T, e, rid);
    new_marks |= after << (8 * r);
    bool was = before & 1u, now = after & 1u;
    int delta = __popc(after) - __popc(before);  // sum(goals_before) - sum(goals_after)
    double v = 0.0;
    v = __dadd_rn(v, __dmul_rn((double)delta, T.r_node));
    v = __dadd_rn(v, (now && !was) ? T.r_recipe : 0.0);
    v = __dadd_rn(v, (!now && was) ? T.r_penalty : 0.0);
    v = __dadd_rn(v, T.r_time);
    all_done = all_done && now;
    any_done = any_done || now;
    // which agent is the r-th relevant one?
    uint32_t m = relevant;
#pragma unroll 1
    for (int q = 0; q < r; ++q) m &= m - 1;
    if (m) reward[__ffs(m) - 1] = v;
  }
  e.marks = new_marks;
  const bool done = T.end_all ? all_done : any_done;
  int k = 0;
  for (int i = 0; i < A; ++i) {
    bool rel = relevant >> i & 1u;
    if (!rel || k >= T.R) reward[i] = 0.0;
    if (rel) ++k;
    term_out[i] = (rel && done) ? 1 : 0;
    trunc_out[i] = (trunc_mask >> i & 1u) ? 1 : 0;
    e.ag[i * OSTRIDE] = (e.ag[i * OSTRIDE] & ~(1u << 15)) | ((active >> i & 1u) << 15);
  }
  uint32_t n_live = __popc(relevant);
  e.tinfo = (t & 0xFFFFFu) | ((done || time_up) ? TI_DONE : 0u) | (n_live << 21);
}
