/* cz_b200.h — C ABI of libcz_b200.so, the B200 (sm_100a) batched CookingZoo step path.
 *
 * The reference (DavidRother/cooking_zoo) is pure Python and has no FFI: its boundary for
 * this path is the in-process Python env API.  Each entry point below names the reference
 * interface it replaces (paths relative to /root/reference/cooking_zoo/).  The host side
 * that binds these (ctypes) is cooking_zoo_b200/_native.py; the stub a reference maintainer
 * would add is shown in INTEGRATION.md.
 *
 * Conventions: plain pointers and sizes only (no torch / C++ types); every function returns
 * 0 on success or a negative CZ_E* code and cz_last_error() then describes it; no exception
 * crosses the boundary; all env buffers are caller-owned DEVICE memory (cz_*_host variants
 * take HOST memory); launches are asynchronous on the given stream (a cudaStream_t passed
 * as void*, NULL = legacy default stream) with no hidden synchronisation; the library owns
 * only cz_tables.  One host thread per device; not thread-safe on the same state.
 */
#ifndef CZ_B200_H
#define CZ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CZ_ABI_VERSION 2

/* compile-time capacity of the kernels */
#define CZ_MAX_CELLS 64       /* width<=8, height<=8; device cell index = y*8 + x */
#define CZ_MAX_DYN 32         /* dynamic-object slots (sum of meta counts of dynamic types) */
#define CZ_MAX_AGENTS 4
#define CZ_MAX_RECIPES 4      /* recipes evaluated per environment */
#define CZ_MAX_NODES 8        /* nodes per recipe (Recipe.node_list) */
#define CZ_MAX_TYPES 16       /* dynamic types */
#define CZ_MAX_STATIC_SLOTS 96
#define CZ_MAX_SPECIAL 4      /* cutboards / blenders / switches / blocks per level (each) */

/* error codes */
#define CZ_OK 0
#define CZ_EINVAL (-1)
#define CZ_ECUDA (-2)
#define CZ_ELIMIT (-3)

/* per-environment error_flags bits: "the reference would have raised / diverged here" */
#define CZ_ERR_CUTBOARD_NONE 1u   /* Cutboard.action() returns None (world_objects.py:250-269)      */
#define CZ_ERR_REMOVE 2u          /* list.remove of an object not in content (cooking_world.py:254) */
#define CZ_ERR_SWITCH_LINK 4u     /* Switch linked to a Switch: no switch_state (world_objects.py:165-169) */
#define CZ_ERR_SPAWN_LOC 8u       /* generate_location timed out (parsing.py:154-167)               */
#define CZ_ERR_TRUNC_DESPAWN 16u  /* IndexError at cooking_env.py:348 (truncation with despawned agent) */
#define CZ_ERR_OBS_OVERFLOW 32u   /* more objects of a type than meta slots (cooking_env.py:371)    */
#define CZ_ERR_OFFGRID 64u        /* scheme1 INTERACT_PRIMARY / EXECUTE_ACTION facing a cell off the grid: get_objects_at(...)[0]
                                     IndexError (cooking_world.py:119, :160); PICK_UP_SPECIAL there is a silent no-op (:138-154) */
#define CZ_ERR_BAD_ID 128u        /* cz_reset: layout id / recipe id outside the compiled tables (id 0 was used instead) */

/* ---- packed per-environment state --------------------------------------------------
 * `state` is a u32 matrix [cz_state_rows()][n_envs] (structure of arrays: row-major, the
 * environment index is the fastest axis).  Rows:
 *   [0, D)          dynamic-object slot records   (D = num_dyn_slots, canonical meta order)
 *   [D, D+A)        agent records                 (A = num_agents)
 *   D+A+0  SBITS    mutable bits of static objects
 *   D+A+1  TINFO    bits 0-19 t | 20 done | 21-23 n_live | 24-31 reserved
 *   D+A+2  MARKS    recipe r: bits [8r, 8r+8) = node_list[k].marked
 *   D+A+3  VARIANT  static variant id of the current layout
 *   D+A+4  RECIPES  recipe r: bits [8r, 8r+8) = index into the compiled recipe list
 *   D+A+5  EPISODE  episodes started by this environment (auto-reset counter)
 *
 * object record : 0-2 x | 3-5 y | 6 present | 7 chopped | 8 mashed | 9 free |
 *                 10-11 container kind (0 held by agent, 1 static content, 2 plate content) |
 *                 12-16 container id (agent index / 0 / plate slot) | 17-22 position in content |
 *                 23-29 Plate records only: number of items on the plate (len(plate.content))
 * agent record  : 0-2 x | 3-5 y | 6-8 orientation | 9 holding? | 10-14 held slot |
 *                 15 active | 16-31 grace period left
 * SBITS         : 0-3 cutboard k READY | 4-7 blender k READY | 8-11 blender k toggle |
 *                 12-15 switch k active | 16-19 block k walkable
 */
#define CZ_ROW_SBITS 0
#define CZ_ROW_TINFO 1
#define CZ_ROW_MARKS 2
#define CZ_ROW_VARIANT 3
#define CZ_ROW_RECIPES 4
#define CZ_ROW_EPISODE 5
#define CZ_NUM_MISC_ROWS 6

/* cz_step flags */
#define CZ_STEP_AUTO_RESET 1u  /* an environment whose `done` bit is set is re-initialised from
                                  the layout pool instead of stepped (reward 0, flags 0) */
#define CZ_STEP_OBS_F32 2u     /* `obs` points to float32 [n][A][L]: each element is the float64
                                  observation rounded to float32 (the reference's obs.astype(float32));
                                  honoured by cz_step, cz_step_pipelined and cz_step_host */
#define CZ_STEP_DEVICE_ACTIONS 4u /* cz_step ignores `actions` (may be NULL) and draws step k's actions on the device from the
                                  counter stream of cz_random_actions at step index action_step + k */
#define CZ_STEP_KEEP_ALL 8u    /* cz_step with k_steps > 1: obs / reward / terminated / truncated are [k_steps][...] arrays and
                                  every step's outputs are kept; without it each step overwrites the same [n][A][...] buffers */
#define CZ_STEP_EPISODE_STATS 16u /* update the episode statistics attached with cz_stats_attach after every step of every
                                  environment (honoured by cz_step, cz_step_pipelined and cz_step_host; CZ_EINVAL when no
                                  statistics are attached or their n_envs differs from the call's) */

/* ---- episode statistics ----------------------------------------------------------------------
 * Every environment carries a record (cz_stats_desc).  After each step of the environment, with the post-step rows EPISODE,
 * TINFO (t, done) and MARKS and that step's rewards r[a]:
 *   1. EPISODE != episode: a reset happened since the last step (cz_reset, masked or not, or an auto-reset step):
 *      episode = EPISODE, ret[:] = 0, open = 1.
 *   2. open: ret[a] = ret[a] + r[a] for every agent (float64, round to nearest, in step order).
 *   3. open and TINFO's done bit: the episode just finished.  last_ret = ret, last_len = t, last_served = number of the R
 *      recipes whose root mark (bit 0 of MARKS byte r) is set, last_success = the recipe condition of
 *      end_condition_all_dishes (all R recipes if set, any if not; a time-up alone gives 0), finished += 1,
 *      totals += (1, t, served, success, ret[0..A)), open = 0.
 * An auto-reset step has reward 0 and leaves t = 0, so it adds nothing; without auto-reset a finished environment that keeps
 * stepping is counted once.  The record keeps only the LAST finished episode: when one call of K steps can finish several
 * episodes of an environment, read the totals.
 * totals f64 [4 + A]: episodes, sum of lengths, recipes served, successes, then the return sum of each agent.  The first four
 * are integers held exactly; the return sums are added per block and then across blocks with atomics, so their last bits
 * depend on the summation order (run to run they may differ by rounding; the per-environment fields never do). */
typedef struct cz_stats_desc {
  int32_t n_envs;
  double* ret;             /* [n][A] return of the running episode                                   */
  uint32_t* episode;       /* [n] internal: EPISODE row the record has seen last                     */
  uint8_t* open;           /* [n] internal: the running episode is being counted                     */
  double* last_ret;        /* [n][A] return of the last finished episode                             */
  int32_t* last_len;       /* [n] its length (t at done)                                             */
  uint8_t* last_served;    /* [n] its recipes served                                                 */
  uint8_t* last_success;   /* [n] its recipe condition (0 / 1)                                       */
  int32_t* finished;       /* [n] episodes finished since cz_stats_clear                             */
  double* totals;          /* [4 + A] sums since cz_stats_clear (layout above)                       */
} cz_stats_desc;

/* Host-side description of everything compiled once per (level, meta, recipes, scheme):
 * replaces load_level.load_level / parsing.parse_* (engine/load_level.py:55-71,
 * engine/parsing.py:5-151), the class tables of world_objects.py, recipe_drawer.py:40-118
 * and the constructor of CookingEnvironment (environment/cooking_env.py:62-161).
 * All pointers are HOST memory, copied by cz_tables_create. */
typedef struct cz_table_desc {
  int32_t abi_version;
  int32_t width, height;
  int32_t num_agents;         /* A: agents per environment                                  */
  int32_t num_recipes;        /* R: recipes evaluated per environment (>= A in the reference) */
  int32_t num_dyn_slots;      /* D */
  int32_t num_static_slots;   /* S: observed static slots (meta order)                      */
  int32_t num_types;          /* dynamic types                                              */
  int32_t num_comp_slots;     /* entries of comp_slots                                      */
  int32_t num_obs_segs;       /* table segments of an observation row (0..2)                */
  int32_t num_obs_ranges;     /* computed ranges of an observation row (1..3)               */
  int32_t obs_table_len;      /* doubles per (variant, cell) entry of obs_table             */
  int32_t obs_segs[2][3];     /* {row offset, length, table offset} in doubles, all even    */
  int32_t obs_ranges[3][2];   /* {row offset, length} of the computed parts of a row        */
  int32_t obs_len;            /* L: doubles per agent observation                           */
  int32_t num_variants;       /* V: distinct static configurations in the layout pool       */
  int32_t num_layouts;        /* P: layout pool size                                        */
  int32_t num_book;           /* B: compiled recipes                                        */
  int32_t max_steps;
  int32_t end_all;            /* end_condition_all_dishes                                   */
  int32_t action_scheme;      /* 1 or 3 (ActionScheme1 / ActionScheme3, cooking_world/actions.py)  */
  int32_t grace_period;
  int32_t num_switches, num_blocks;
  double reward_node, reward_recipe, reward_penalty; /* reward_scheme terms                  */
  double reward_time;         /* max_time_penalty / max_steps, divided by the host           */
  double respawn_rate, despawn_rate;
  const double* xlut;         /* [2*width-1]  k/width  for k=-(width-1)..width-1            */
  const double* ylut;         /* [2*height-1]                                               */
  const uint8_t* grid;        /* [V][64] low nibble static kind, high nibble special index  */
  const uint8_t* static_cells;/* [V][S] cell of observed static slot, 0xFF = empty          */
  const uint8_t* scan_order;  /* [V][D] dynamic slots in get_objects_at scan order          */
  const uint8_t* special_cells;/* [V][4 kinds][CZ_MAX_SPECIAL] cell, 0xFF = none            */
  const uint64_t* static_masks;/* [V][8] cells occupied by each static kind                 */
  const uint8_t* slot_type;   /* [D] dynamic type id of a slot                              */
  const uint8_t* type_flags;  /* [T] 1 plate | 2 chop | 4 blend | 8 spawn-on-chop           */
  const uint8_t* type_base;   /* [T] first slot of the type                                 */
  const uint8_t* type_count;  /* [T] slots of the type                                      */
  const uint32_t* comp_slots; /* [num_comp_slots] 0-11 row offset | 12-14 features after x,y |
                                 15-16 kind (0 static, 1 dynamic, 2 agent) | 17-24 index    */
  const double* obs_table;    /* [V][64][obs_table_len] static parts of a row per observer cell */
  const uint32_t* recipe_nodes;/* [B][8] 0-7 type | 8 static? | 9-10 cond | 16-23 children  */
  const uint8_t* recipe_len;  /* [B] nodes in the recipe                                    */
  const uint32_t* pool;       /* [P][rows] initial state of every pooled layout             */
  const uint8_t* default_recipes; /* [R] recipe index per slot when no per-env ids are given */
  const uint8_t* spawn_x;     /* [A][8] X_POSITION list of the agent's spawn entry (parsing.py:147)  */
  const uint8_t* spawn_y;     /* [A][8] Y_POSITION list                                      */
  const uint8_t* spawn_n;     /* [A][2] lengths of the two lists                             */
  const uint64_t* layout_cum; /* [P] or NULL.  Weighted pool (the exact layout distribution of the reference's level
                                 parser, engine/parsing.py:21-151): cumulative probabilities scaled to 2^64; a 64-bit
                                 draw u selects the first layout with layout_cum[i] > u.  NULL: uniform pool, u % P. */
} cz_table_desc;

typedef struct cz_tables cz_tables;

/* Compile-once tables -> device.  Replaces CookingWorld.__init__ + load_level + the class
 * and recipe tables (cooking_world/cooking_world.py:23-44, 263-265). */
int cz_tables_create(const cz_table_desc* desc, int device, cz_tables** out);
int cz_tables_destroy(cz_tables* t);

/* Rows of the u32 state matrix for these tables (= D + A + CZ_NUM_MISC_ROWS). */
int cz_state_rows(const cz_tables* t);

/* CookingEnvironment.reset (environment/cooking_env.py:178-210) for every environment whose
 * mask byte is non-zero (mask NULL = all): copy pooled layout layout_ids[e] into the state,
 * evaluate the recipes (cooking_book/recipe.py:77-87), write the first observations
 * (cooking_env.py:352-373).  recipe_ids: [n][R] u8 or NULL (default assignment).  An id outside the
 * compiled tables is replaced by 0 and reported as CZ_ERR_BAD_ID in error_flags (u32 [n], may be NULL). */
int cz_reset(const cz_tables* t, uint32_t* state, const int32_t* layout_ids, const uint8_t* recipe_ids,
             const uint8_t* mask, double* obs, uint32_t* error_flags, int n_envs, void* stream);

/* layout_ids[e] = cz_layout_index(t, seed, env_offset + e, episode) on the device: the default layout of
 * every environment's `episode`-th episode, the same draw CZ_STEP_AUTO_RESET makes. */
int cz_layout_ids(const cz_tables* t, int32_t* layout_ids, int n_envs, uint64_t seed, int64_t env_offset,
                  uint64_t episode, void* stream);

/* CookingEnvironment.accumulated_step + observe (environment/cooking_env.py:243-288), k_steps times:
 * world_step (cooking_world/cooking_world.py:104-112, action_scheme3.py:4-43), compute_rewards /
 * compute_truncated (:290-350), get_feature_vector (:352-373) for n_envs environments.
 * actions u8 [k_steps][n][A] (0..4 under scheme3, 0..7 under scheme1); obs f64 [n][A][L]; reward f64 [n][A];
 * terminated/truncated u8 [n][A] (each with a leading [k_steps] axis under CZ_STEP_KEEP_ALL);
 * error_flags u32 [n] (OR-accumulated, may be NULL).  With CZ_STEP_AUTO_RESET the layout of
 * episode k of global environment g = env_offset + e is pool[cz_layout_index(t, seed, g, k)].
 * k_steps > 1 (and single steps of small batches) run as ONE launch of the warp-per-environment kernel
 * (csrc/cz_warp.cuh: the environment stays in registers between steps, rows stream out after every step)
 * when the tables are in the specialised class; otherwise as k_steps launches of the per-step kernels.
 * The results do not depend on which kernel ran. */
int cz_step(const cz_tables* t, uint32_t* state, const uint8_t* actions, double* obs, double* reward,
            uint8_t* terminated, uint8_t* truncated, uint32_t* error_flags, int n_envs, int k_steps,
            uint32_t flags, uint64_t seed, int64_t env_offset, uint64_t action_step, void* stream);

/* Attach caller-owned device buffers for CZ_STEP_EPISODE_STATS (NULL detaches).  Every pointer is required and n_envs >= 1,
 * or CZ_EINVAL.  The tables keep the pointers, not the buffers: they must outlive the attachment. */
int cz_stats_attach(cz_tables* t, const cz_stats_desc* desc);
/* Start a counting window (one small kernel on `stream`): ret, the last_* fields, finished and the totals become 0,
 * episode = EPISODE and open = (t == 0), so an episode that has not taken a step yet is counted whole and one already
 * running is not counted at all. */
int cz_stats_clear(const cz_tables* t, const uint32_t* state, int n_envs, void* stream);

/* get_feature_vector only (cooking_env.py:352-373): rebuild obs from the current state. */
int cz_observe(const cz_tables* t, const uint32_t* state, double* obs, int n_envs, void* stream);

/* The same rows as float32 (element-wise rounding of the float64 rows; any observation plan).
 * cz_reset and cz_step accept obs == NULL (state / rewards / flags only), so a float32 consumer never
 * pays for float64 rows: cz_reset(..., NULL, ...) + cz_observe_f32, then cz_step with CZ_STEP_OBS_F32. */
int cz_observe_f32(const cz_tables* t, const uint32_t* state, float* obs32, int n_envs, void* stream);

/* ---- grid observation ----------------------------------------------------------------------
 * Per-cell u8 planes of every agent's world: grid u8 [n][A][C][H][W], cell (x, y) at [..., y, x].  A pure function of the
 * packed state (written after cz_reset / cz_step with obs == NULL) that does not depend on the observation plan.  C depends
 * only on the meta file and A.  Channel order for observer a:
 *   [0, 7)   static kinds in ST_* code order: floor, counter, cutboard, blender, deliversquare, switch, block.  1 where that
 *            static stands; floor is every cell of the W x H grid where no other static stands (one-hot on every cell)
 *   [7, 12)  cutboard_ready, blender_ready, blender_on, switch_active, block_walkable: 1 on the static's cell when its SBITS
 *            bit is set
 *   12 + t   n:<Type> for each dynamic type t of the meta file, in meta order (also types without device slots): number of
 *            present objects of the type at the cell, held objects and plate contents included
 *   then     chopped:<Type> for each type with the chop flag, in meta order: how many of them are chopped
 *   then     mashed:<Type> for each type with the blend flag, in meta order: how many of them are mashed
 *   then     on_plate: number of present objects at the cell whose container is a plate (container kind 2)
 *   then     A agent groups g (group 0 = agent a, then the other agents in ascending index), 7 channels each:
 *            agent<g> (position), agent<g>_facing1..4 (orientation 1..4), agent<g>_holding, agent<g>_active; 1 at the agent's
 *            cell.  An inactive agent keeps its position and facing planes.
 * So C = 7 + 5 + T + T_chop + T_blend + 1 + 7 A (46 for the shipped meta with two agents).  Not encoded: the order of
 * contents, free flags, grace periods, the clock and recipe marks. */
int cz_grid_channels(const cz_tables* t);
/* grid of every environment from the current state, asynchronous on `stream`; no alignment requirement on `grid`. */
int cz_observe_grid(const cz_tables* t, const uint32_t* state, uint8_t* grid, int n_envs, void* stream);

/* The reference-facing call with HOST buffers: copies actions host->device, steps, copies
 * obs/reward/flags device->host, and synchronises the stream before returning.  Scratch
 * device buffers are owned by the tables object (sized on first use). */
int cz_step_host(cz_tables* t, uint32_t* state_dev, const uint8_t* actions_host, double* obs_host,
                 double* reward_host, uint8_t* terminated_host, uint8_t* truncated_host,
                 int n_envs, uint32_t flags, uint64_t seed, int64_t env_offset, void* stream);

/* The counter-based draw used by auto-reset (splitmix64 finaliser over seed, env, episode). */
uint64_t cz_layout_draw(uint64_t seed, uint64_t global_env, uint64_t episode);

/* Pool index that draw selects under these tables: the first i with layout_cum[i] > draw for a weighted pool,
 * draw % P for a uniform one.  What CZ_STEP_AUTO_RESET and cz_layout_ids compute on the device. */
int cz_layout_index(const cz_tables* t, uint64_t seed, uint64_t global_env, uint64_t episode);

/* Randomness of handle_agent_spawn (cooking_world/cooking_world.py:267-290).  The reference draws
 * np.random.random() for despawn/respawn and random.sample(list, 1) for the respawn cell from
 * global generators; here the c-th draw consumed by environment g in step t of its episode is the
 * uniform double cz_spawn_uniform(seed, g, episode, t, c) in [0, 1), and a list pick is
 * list[floor(u * len)].  Parity harnesses patch the reference's call sites to read this stream. */
double cz_spawn_uniform(uint64_t seed, uint64_t global_env, uint64_t episode, uint64_t t, uint64_t c);

/* Pipelined throughput mode (specialised kernels only).  `state2` is TWO state matrices back to back
 * ([2][rows][n]; more after cz_pipeline_config); step k+1's dynamics (cooking_world.world_step + compute_rewards) run on an internal
 * high-priority stream reading one half and writing the other, while the observation writer
 * (get_feature_vector) of step k is still streaming out on a second internal stream.  Every step does
 * the full work of cz_step; only the ordering guarantee changes: the caller's stream is ordered after the
 * DYNAMICS of the step (state, rewards and flags are final, the action buffer may be overwritten or freed by
 * later work on that stream); the observation rows are ordered with the caller's stream after
 * cz_pipeline_wait().  `actions` must not be modified by any OTHER stream until then.
 * cz_pipeline_reset(t, h) drains the internal streams (host-synchronising) and declares that half h holds
 * the current state; call it BEFORE cz_reset writes into that half. */
int cz_step_pipelined(cz_tables* t, uint32_t* state2, const uint8_t* actions, double* obs, double* reward,
                      uint8_t* terminated, uint8_t* truncated, uint32_t* error_flags, int n_envs,
                      uint32_t flags, uint64_t seed, int64_t env_offset, void* stream);
/* Ring size and background dynamics of the pipelined step (call while nothing is in flight; it drains like
 * cz_pipeline_reset and selects buffer 0).  n_buffers (2..4): `state2` then holds that many state matrices and the dynamics
 * may run n_buffers - 1 steps ahead of the row writer.  dyn_blocks_per_sm (0..8, 0 = full grid): the dynamics kernel is
 * launched with that many blocks per SM and loops over its tiles, so it runs in the background of the row writer of the
 * previous step(s) instead of displacing it — right for open-loop action streams (the step's latency grows), wrong when
 * the next actions depend on this step's state. */
int cz_pipeline_config(cz_tables* t, int n_buffers, int dyn_blocks_per_sm);
int cz_pipeline_wait(cz_tables* t, void* stream);
/* Order the caller's stream after the latest dynamics only (state, rewards, flags are final; the observation
 * rows of that step may still be streaming out): what a device policy reading the state needs. */
int cz_pipeline_wait_state(cz_tables* t, void* stream);
int cz_pipeline_reset(cz_tables* t, int current_half);
int cz_pipeline_current(const cz_tables* t);

/* ---- Scripted cook as a device policy (SURVEY.md §8 f3) -----------------------------------
 * Replaces CookingAgent.step (cooking_agents/cooking_agent.py:9-122) + BaseAgent.walk_to_location /
 * reachable / closest / generic_sequence (cooking_agents/base_agent.py:49-199), which the reference
 * evaluates per agent on a deep-copied symbolic observation.  The decision is a pure function of the
 * world, so the policy keeps no state; its two graph searches over the Floor tiles are host-built
 * tables per static variant (cooking_zoo_b200/policy.py). */
typedef struct cz_policy_desc {
  int abi_version;
  int num_variants;           /* must equal cz_table_desc.num_variants                          */
  const uint8_t* lists;       /* [V][8 static kinds][64] cells of each static kind (Floor, Counter,
                                 Cutboard, ...) in world_objects list order                      */
  const uint8_t* list_len;    /* [V][8]                                                          */
  const uint64_t* reach;      /* [V][64] bit b of reach[a]: BaseAgent.reachable(a, b)            */
  const uint8_t* first_step;  /* [V][64 from][64 to] action 0..4 of BaseAgent.walk_to_location   */
} cz_policy_desc;

typedef struct cz_policy cz_policy;
int cz_policy_create(const cz_tables* t, const cz_policy_desc* desc, cz_policy** out);
int cz_policy_destroy(cz_policy* p);
/* blocks_per_sm > 0: cz_policy_act launches that many blocks per SM and walks the batch in strides (a background policy
 * for the pipelined closed loop: it shares the SMs with the row writer of the previous step instead of displacing it);
 * 0 (default): one thread per environment in one wave. */
int cz_policy_config(cz_policy* p, int blocks_per_sm);

/* One CookingAgent.step per agent of every environment, on the CURRENT state.
 * cook_recipes u8 [n][A]: recipe-book index each cook follows, or NULL (cook i follows recipe i of
 * its environment).  actions u8 [n][A] (0..4: the cook only ever walks).  crashed u8 [n] (may be
 * NULL): bit i set where the reference cook would raise (no object of the wanted type, nothing
 * reachable; oracle/cz_policy.py lists the sites) — that agent's action is 0.
 * Ordered on `stream` like every other call.  While a pipelined run is in flight (cz_step_pipelined has been called since
 * the last cz_pipeline_reset) the kernel itself runs on the library's high-priority dynamics stream, fenced by events
 * before and after, so that it does not queue behind the row writer of the previous step (closed loop, one CUDA graph of
 * 40 steps: 138.4 -> 123.0 us per step); CZ_POLICY_ON_DYN=0 in the environment of cz_tables_create switches that off. */
int cz_policy_act(const cz_policy* p, const uint32_t* state, const uint8_t* cook_recipes, uint8_t* actions,
                  uint8_t* crashed, int n_envs, void* stream);

/* Synthetic action streams generated on the device (SURVEY.md §8d, configs 3 and 4: uniform random actions):
 * actions[e][i] = floor(u * len(ACTIONS)) with u = cz_spawn_uniform(seed ^ 0xA5A5A5A5A5A5A5A5, env_offset + e, 0, step, i),
 * len(ACTIONS) = 5 under scheme3, 8 under scheme1 (cooking_world/actions.py:2-17, 39-50).  Counter-based: the stream
 * of an environment does not depend on the batch it is stepped in. */
int cz_random_actions(const cz_tables* t, uint8_t* actions, int n_envs, uint64_t seed, uint64_t step,
                      int64_t env_offset, void* stream);

/* Number of kernels launched by this library since load (the bench's gpu_launches claim). */
uint64_t cz_launch_count(void);

const char* cz_last_error(void);
int cz_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* CZ_B200_H */
