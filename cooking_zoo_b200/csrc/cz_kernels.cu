// cz_kernels.cu — kernels and the C ABI of libcz_b200.so (sm_100a only).
//
// Execution model ("tile" = 32 consecutive environments owned by one warp):
//   1. the warp loads the tile's packed state, structure-of-arrays in HBM, into shared-memory
//      columns with coalesced 128 B loads (lane = environment);
//   2. every lane advances its environment one step (cz_device.cuh) — scalar table-driven
//      code, no cross-lane traffic;
//   3. state, rewards and flags go back with coalesced stores;
//   4. the warp walks its 32 x A observation rows: the lanes fill one row (one lane per
//      observed slot) in a shared-memory staging buffer and a single elected lane hands the
//      2224-byte row to the TMA engine (cp.async.bulk shared->global, SASS UBLKCP), double
//      buffered so row r+1 is built while row r drains.
// The path is HBM-write bound (observations are 92 % of the bytes); tensor cores are unused.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <new>

#include "cz_device.cuh"

#ifndef CZ_WARPS_PER_BLOCK
#define CZ_WARPS_PER_BLOCK 4
#endif
#define CZ_THREADS (32 * CZ_WARPS_PER_BLOCK)
#ifndef CZ_DYN_MIN_BLOCKS
#define CZ_DYN_MIN_BLOCKS CZ_MIN_BLOCKS  // the dynamics-only instantiation (OBS_NONE) of the pipelined step
#endif
#ifndef CZ_MIN_BLOCKS
#define CZ_MIN_BLOCKS (28 / CZ_WARPS_PER_BLOCK)  // 28 warps/SM: registers capped at 72, shared memory at 32 KB per block
#endif

enum { MODE_STEP = 0, MODE_RESET = 1, MODE_OBSERVE = 2 };
#define CZ_FLAG_TILE_SHIFT 8  // internal bits 8-10 of the kernel's `flags`: log2(environments per warp)
enum { OBS_TMA = 0, OBS_STG = 1, OBS_NONE = 2 };  // OBS_NONE: dynamics only (pipelined step: the observe kernel follows)
#ifndef CZ_STAGE_SETS
#define CZ_STAGE_SETS 1  // sets of staging rows per warp (2 = double buffered; measured: no gain, profiles/r01_notes.md)
#endif

// ---- Ampere-style async copies (LDGSTS) for the 4-byte state words -------------------------
__device__ __forceinline__ void cz_cp_async4(void* sdst, const void* gsrc) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(sdst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cz_cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---- TMA bulk store helpers (PTX ISA: cp.async.bulk, sm_90+) ------------------------------
__device__ __forceinline__ void cz_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void cz_bulk_store_nocommit(void* gdst, const void* ssrc, uint32_t bytes) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes) : "memory");
}
// The same with an L2 evict_first hint, for writers whose WHOLE output block leaves in one bulk store (nothing else writes
// into its 128-byte lines later and nothing on the device reads it back): 131072 envs, float32 pair writer 52.0 -> 44.4 us.
// On the float64 packed writer, whose table segments are lane stores into the same lines, the hint loses (94.1 -> 102.8 us).
#ifndef CZ_BULK_STREAM_HINT
#define CZ_BULK_STREAM_HINT 1
#endif
__device__ __forceinline__ void cz_bulk_store_stream(void* gdst, const void* ssrc, uint32_t bytes) {
#if CZ_BULK_STREAM_HINT
  uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst), "r"(s), "r"(bytes), "l"(pol) : "memory");
#else
  cz_bulk_store_nocommit(gdst, ssrc, bytes);
#endif
}
__device__ __forceinline__ void cz_bulk_store_s(void* gdst, uint32_t ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cz_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cz_bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

// Row stores of the warp-per-environment writer.  CZ_OBS_ST selects the cache operator (A/B builds through
// CZ_NVCC_EXTRA=-DCZ_OBS_ST=1|2): 0 default (write-back), 1 st.global.cs (streaming, evict first), 2 st.global.wt.
#ifndef CZ_OBS_ST
#define CZ_OBS_ST 0
#endif
__device__ __forceinline__ void cz_row_store(double2* p, const double2 v) {
#if CZ_OBS_ST == 1
  __stcs(p, v);
#elif CZ_OBS_ST == 2
  __stwt(p, v);
#else
  *p = v;
#endif
}

// ---- observation rows (get_feature_vector, cooking_env.py:352-373) -----------------------------
// A row = table segments (static slots: a function of layout variant and observer cell only, copied
// from the L2-resident obs_table with 128-bit loads/stores) + computed slots (dynamic objects,
// agents, live Switch/Block) written as [x, y, flags..., 1] doubles into shared-memory staging rows
// that the TMA engine stores (cp.async.bulk).  Slots that can never be occupied are not listed: the
// staging rows are zero-filled once and only the listed slots are rewritten.
//
// Everything that does not change from row to row is decoded once per kernel into LaneSlot.  In the
// FAST instantiation a lane owns one (observer, slot) pair, so all A rows of an environment are
// filled in a single pass; otherwise a lane owns one slot and loops over the observers.
struct LaneSlot {
  int off;        // staging offset (doubles, inside its row) of the slot owned by this lane, < 0: idle
  int agent;      // FAST: the observer (row) this lane writes
  uint32_t flen;  // features after x, y (the trailing 1 included)
  uint32_t kind;  // 0 live static (Switch/Block), 1 dynamic object, 2 agent
  uint32_t idx;   // static slot / dynamic slot / agent index
  int t0, t1;     // destination (double2 units, relative to the row) of table elements lane, lane+32
};

__device__ __forceinline__ LaneSlot cz_lane_slot(const CzDev& T, int q, int agent, int lane) {
  LaneSlot ls;
  ls.off = -1; ls.agent = agent; ls.flen = 1; ls.kind = 1; ls.idx = 0;
  if (q >= 0 && q < T.n_comp) {
    const uint32_t d = __ldg(T.comp_slots + q);
    ls.off = (int)(d & 0xFFFu) - T.stage_lo;
    ls.flen = (d >> 12) & 7u; ls.kind = (d >> 15) & 3u; ls.idx = (d >> 17) & 255u;
  }
  // table element k (double2 units) -> row position: segment 0 first, then segment 1
  const int n0 = T.n_segs > 0 ? T.segs[0][1] >> 1 : 0, n1 = T.n_segs > 1 ? T.segs[1][1] >> 1 : 0;
  ls.t0 = ls.t1 = -1;
  int k = lane;
  if (k < n0) ls.t0 = (T.segs[0][0] >> 1) + k; else if (k < n0 + n1) ls.t0 = (T.segs[1][0] >> 1) + k - n0;
  k = lane + 32;
  if (k < n0) ls.t1 = (T.segs[0][0] >> 1) + k; else if (k < n0 + n1) ls.t1 = (T.segs[1][0] >> 1) + k - n0;
  return ls;
}

// The same from the host-prepared per-lane maps (packed (observer, slot) layout of the specialised kernels).
__device__ __forceinline__ LaneSlot cz_lane_slot_packed(const CzDev& T, int lane) {
  LaneSlot ls;
  const int4 lm = __ldg(T.lane_map + lane);
  ls.off = -1; ls.agent = lm.y; ls.flen = 1; ls.kind = 1; ls.idx = 0;
  if (lm.x >= 0) {
    const uint32_t d = (uint32_t)lm.x;
    ls.off = (int)(d & 0xFFFu) - T.stage_lo;
    ls.flen = (d >> 12) & 7u; ls.kind = (d >> 15) & 3u; ls.idx = (d >> 17) & 255u;
  }
  ls.t0 = lm.z;
  ls.t1 = lm.w;
  return ls;
}

// Observer-independent part of a computed slot: cell (x | y<<3, bit 6 = present) and feature bits.
// Agent columns follow the object columns in shared memory, so dynamic objects and agents are
// decoded by the same instruction stream (no divergence between the two kinds of lane).
template <bool FAST>
__device__ __forceinline__ void cz_slot_state(const CzDev& T, const SmemTabs* st, const LaneSlot& ls,
                                              const uint32_t* sobj, const uint32_t* sag, uint32_t sbits,
                                              uint32_t variant, int e, uint32_t& xy, uint32_t& fb) {
  uint32_t rec, fb4;
  bool present;
  if (ls.kind != 0) {
    // dynamic object: [!done, chopped, mashed] (world_objects.py:447,555,...);
    // agent: one-hot orientation; every agent, active or not (cooking_env.py:356)
    const bool is_agent = ls.kind == 2;
    const bool exists = !is_agent || (int)ls.idx < T.A;
    rec = exists ? (is_agent ? sag : sobj)[ls.idx * OSTRIDE + e] : 0u;
    present = is_agent ? exists : (rec & O_PRESENT) != 0;
    const uint32_t c = (rec >> 7) & 1u, m = (rec >> 8) & 1u;
    fb4 = is_agent ? ((1u << A_ORI(rec)) >> 1) : (((c | m) ^ 1u) | c << 1 | m << 2);
  } else {  // live Switch / Block: [switch_active] / [walkable] (world_objects.py:174,221)
    uint32_t cell = TAB_SCELL(variant, ls.idx);
    present = cell != 0xFFu;
    rec = present ? cell : 0u;
    uint32_t g = TAB_GRID(variant, rec);
    fb4 = ((g & 15u) == ST_SWITCH ? (sbits >> (12 + (g >> 4))) : (sbits >> (16 + (g >> 4)))) & 1u;
  }
  const uint32_t one = 1u << (ls.flen - 1);  // the trailing 1 of every feature vector
  fb = present ? ((fb4 & (one - 1u)) | one) : 0u;
  xy = (rec & 63u) | (present ? 64u : 0u);
}

// Observer-dependent part: (x - ax) / W, (y - ay) / H from shared tables of host-divided doubles
// (the observer's own entry is x / W, y / H: cooking_env.py:364-368), then the flags as doubles
// (1.0 = 0x3FF00000'00000000).
__device__ __forceinline__ void cz_slot_store(const LaneSlot& ls, uint32_t xy, uint32_t fb, int ax, int ay, bool self,
                                              const double* sxl, const double* syl, double* row) {
  const int x = xy & 7u, y = (xy >> 3) & 7u;
  double X = sxl[x - (self ? 0 : ax)];
  double Y = syl[y - (self ? 0 : ay)];
  if (!(xy & 64u)) { X = 0.0; Y = 0.0; }
  double* out = row + ls.off;
  out[0] = X;
  out[1] = Y;
#pragma unroll
  for (int k = 0; k < 5; ++k)
    if (k < (int)ls.flen) *reinterpret_cast<uint2*>(out + 2 + k) = make_uint2(0u, (fb >> k & 1u) ? 0x3FF00000u : 0u);
}

// per-warp words: object columns [D][33], agent columns [A][33], then sbits/variant/wobs [32]
struct WarpSmem {
  uint32_t* obj;
  uint32_t* ag;
  uint32_t* sbits;
  uint32_t* variant;
  uint32_t* wobs;
};

// Observation phase of the specialised kernels (NA agents known at compile time; one lane per
// (observer, slot) pair; one computed range; at most 64 table double2 per row).
// Software pipeline over the tile's environments: the table segments of environment le+1 are
// requested (LDG) right after environment le's staging rows were handed off and are stored one
// iteration later, so neither the L2 latency nor the proxy fence's drain sits on the critical path.
// OBS_TMA: the staging rows are double buffered (NBUF sets of NA rows) and go out through the TMA
// engine; OBS_STG: the lanes copy them out with 128-bit stores.
template <int NA, int OBS>
__device__ __forceinline__ void cz_obs_phase_fast(const CzDev& T, const SmemTabs* st, const WarpSmem* ws, const double* sxl,
                                                  const double* syl, double* stage, uint32_t stage_s, int row_stride,
                                                  uint32_t row_bytes, double* genv, int n_here, int lane, int tab2, int L2,
                                                  size_t row_gbytes, uint32_t r0_bytes, size_t r0_goff, uint32_t r0_soff) {
  constexpr int NP = NA < 2 ? NA : 2;  // rows whose table segments are prefetched
  const LaneSlot ls = cz_lane_slot_packed(T, lane);
  const double2* tab0 = reinterpret_cast<const double2*>(T.obs_table) + lane;
  const size_t var_stride = (size_t)64 * tab2;
  const bool self = ls.kind == 2 && (int)ls.idx == ls.agent;
  const uint32_t* my_me = ws->ag + ls.agent * OSTRIDE;  // the observer of this lane's pair
  const int set_stride = NA * row_stride;               // doubles between the two staging sets
  const int r0_off2 = (int)(r0_goff >> 4), r0_n2 = (int)(r0_bytes >> 4);

  double2 v0[NP], v1[NP];
  {  // prefetch for the first environment
    const double2* tab = tab0 + (size_t)ws->variant[0] * var_stride;
#pragma unroll
    for (int a = 0; a < NP; ++a) {
      const double2* src = tab + (ws->ag[a * OSTRIDE] & 63u) * tab2;
      if (ls.t0 >= 0) v0[a] = __ldg(src);
      if (ls.t1 >= 0) v1[a] = __ldg(src + 32);
    }
  }
  int buf = 0;
#pragma unroll 1
  for (int le = 0; le < n_here; ++le, genv += (size_t)NA * T.L, buf = (buf + 1) % CZ_STAGE_SETS) {
    const bool w = ws->wobs[le] != 0;
    const uint32_t sb = ws->sbits[le], var = ws->variant[le];
    uint32_t xy = 0, fb = 0;
    if (ls.off >= 0) cz_slot_state<true>(T, st, ls, ws->obj, ws->ag, sb, var, le, xy, fb);
    const uint32_t me = my_me[le];
    double* set = stage + (OBS == OBS_TMA ? buf * set_stride : 0);
    // every value of this lane's slot is computed before the synchronisation below (whose memory
    // clobber stops the compiler from hoisting the table loads itself); only stores follow it
    double X, Y;
    uint32_t hi[5];
    {
      const int x = xy & 7u, y = (xy >> 3) & 7u;
      X = sxl[x - (self ? 0 : (int)(me & 7u))];          // (x - ax) / W, or x / W for the observer itself
      Y = syl[y - (self ? 0 : (int)((me >> 3) & 7u))];
      if (!(xy & 64u)) { X = 0.0; Y = 0.0; }
#pragma unroll
      for (int k = 0; k < 5; ++k) hi[k] = (fb >> k & 1u) ? 0x3FF00000u : 0u;  // 1.0 = 0x3FF00000'00000000
    }
    if (OBS == OBS_TMA) {
      // the bulk stores that last read this staging set must have drained
      if (lane == 0) cz_bulk_wait_read<CZ_STAGE_SETS - 1>();
      __syncwarp();
    }
    if (ls.off >= 0) {
      double* out = set + ls.agent * row_stride + ls.off;
      out[0] = X;
      out[1] = Y;
#pragma unroll
      for (int k = 0; k < 5; ++k)
        if (k < (int)ls.flen) *reinterpret_cast<uint2*>(out + 2 + k) = make_uint2(0u, hi[k]);
    }
    if (OBS == OBS_TMA) {
      cz_fence_async_smem();  // generic-proxy writes -> visible to the async proxy
      __syncwarp();
      if (lane == 0 && w) {  // one elected lane hands the computed range of the NA rows to the TMA engine
        char* gp = reinterpret_cast<char*>(genv) + r0_goff;
        uint32_t sp = stage_s + r0_soff + (uint32_t)(buf * set_stride) * 8u;
#pragma unroll
        for (int a = 0; a < NA; ++a, gp += row_gbytes, sp += row_bytes) cz_bulk_store_s(gp, sp, r0_bytes);
      }
      if (lane == 0) cz_bulk_commit();
    } else {
      __syncwarp();
      if (w) {
#pragma unroll
        for (int a = 0; a < NA; ++a) {
          const double2* s2 = reinterpret_cast<const double2*>(set + a * row_stride) + (r0_soff >> 4);
          double2* g2r = reinterpret_cast<double2*>(genv) + a * L2 + r0_off2;
          for (int k = lane; k < r0_n2; k += 32) g2r[k] = s2[k];
        }
      }
      __syncwarp();
    }
    // table segments: rows 0..NP-1 were requested one iteration ago
    double2* g2 = reinterpret_cast<double2*>(genv);
    if (w) {
#pragma unroll
      for (int a = 0; a < NP; ++a) {
        if (ls.t0 >= 0) g2[a * L2 + ls.t0] = v0[a];
        if (ls.t1 >= 0) g2[a * L2 + ls.t1] = v1[a];
      }
#pragma unroll
      for (int a = NP; a < NA; ++a) {  // more than two agents: loaded and stored here
        const double2* src = tab0 + (size_t)var * var_stride + (ws->ag[a * OSTRIDE + le] & 63u) * tab2;
        if (ls.t0 >= 0) g2[a * L2 + ls.t0] = __ldg(src);
        if (ls.t1 >= 0) g2[a * L2 + ls.t1] = __ldg(src + 32);
      }
    }
    if (le + 1 < n_here) {  // request the table segments of the next environment
      const double2* tab = tab0 + (size_t)ws->variant[le + 1] * var_stride;
#pragma unroll
      for (int a = 0; a < NP; ++a) {
        const double2* src = tab + (ws->ag[a * OSTRIDE + le + 1] & 63u) * tab2;
        if (ls.t0 >= 0) v0[a] = __ldg(src);
        if (ls.t1 >= 0) v1[a] = __ldg(src + 32);
      }
    }
  }
  if (OBS == OBS_TMA) {
    if (lane == 0) cz_bulk_wait_read<0>();  // staging and columns are reused by the next tile
  }
}

// Image of the read-only part of a block's shared memory, built on the host (cz_tables_create) and
// copied by every block with one 16-byte load per thread.
struct BlockSmem {
  double xlut[16];  // k / W for k = -(W-1)..W-1
  double ylut[16];
  SmemTabs tabs;
};
__host__ __device__ inline size_t cz_warp_words(int D, int A) { return (size_t)(D + A) * OSTRIDE + 32 * 3; }
// bytes of the image actually used by tables with V static variants (the VarTabs array is the tail of the struct)
__host__ __device__ inline size_t cz_block_smem_head(int V) {
  const int nv = V < 1 ? 1 : (V > CZ_SV ? 1 : V);  // tables with more variants run the generic kernels (global-memory tables)
  return (sizeof(BlockSmem) + (size_t)(nv - 1) * sizeof(VarTabs) + 15) & ~(size_t)15;
}

template <int MODE, int OBS, int NA>
__global__ void __launch_bounds__(CZ_THREADS, OBS == 2 ? CZ_DYN_MIN_BLOCKS : CZ_MIN_BLOCKS)
cz_env_kernel(const __grid_constant__ CzDev T, const uint32_t* state, uint32_t* state_out,  // may alias (in-place step)
              const uint8_t* __restrict__ actions,
              const int32_t* __restrict__ layout_ids, const uint8_t* __restrict__ recipe_ids,
              const uint8_t* __restrict__ mask, double* __restrict__ obs, double* __restrict__ reward,
              uint8_t* __restrict__ term, uint8_t* __restrict__ trunc, uint32_t* __restrict__ errflags,
              int n_envs, uint32_t flags, uint64_t seed, int64_t env_offset, int ld) {
  // `ld`: columns of the state matrix (>= n_envs: a launch may cover a column range of a larger batch, with `state`,
  // the outputs and env_offset already advanced to its first environment)
  // NA = 0: generic kernel (run-time agent count, tables in global memory, any observation plan)
  // NA > 0: specialised kernel for NA agents (tables in shared memory, packed observation lanes)
  constexpr bool FAST = NA != 0;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // lane 0's broadcast tells the compiler the warp index is warp-uniform (uniform datapath, plain UBLKCP operands)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int D = T.D, A = FAST ? NA : T.A;
  BlockSmem* bs = reinterpret_cast<BlockSmem*>(smem_raw);
  WarpSmem wsv;
  WarpSmem* ws = &wsv;
  {
    uint32_t* base = reinterpret_cast<uint32_t*>(smem_raw + cz_block_smem_head(T.V)) + (size_t)warp * cz_warp_words(D, A);
    wsv.obj = base;
    wsv.ag = base + D * OSTRIDE;
    wsv.sbits = wsv.ag + A * OSTRIDE;
    wsv.variant = wsv.sbits + 32;
    wsv.wobs = wsv.variant + 32;
  }
  // staging (the computed span of A rows) lives after the per-warp words, 16-byte aligned
  const size_t row_bytes = ((size_t)T.stage_len * 8 + 15) & ~(size_t)15;
  unsigned char* stage_base = smem_raw + ((cz_block_smem_head(T.V) + cz_warp_words(D, A) * 4 * CZ_WARPS_PER_BLOCK + 15) & ~(size_t)15);
  double* stage = reinterpret_cast<double*>(stage_base + (size_t)warp * CZ_STAGE_SETS * A * row_bytes);
  const int row_stride = (int)(row_bytes >> 3);
  // read-only block image: one 16-byte load per thread
  for (int i = threadIdx.x; i < (int)(cz_block_smem_head(T.V) / 16); i += CZ_THREADS)
    reinterpret_cast<uint4*>(bs)[i] = __ldg(reinterpret_cast<const uint4*>(T.blob) + i);
  // never-occupied slots stay zero: the staging rows are cleared once and only live slots are rewritten
  if (OBS != OBS_NONE)
    for (int i = lane; i < CZ_STAGE_SETS * A * row_stride; i += 32) stage[i] = 0.0;
  const SmemTabs* st = &bs->tabs;
  const double* sxl = bs->xlut + (T.W - 1);
  const double* syl = bs->ylut + (T.H - 1);
  __syncthreads();

  // a tile is 32 environments unless the batch is too small to give every SM scheduler a warp: then the library
  // shrinks it (CZ_FLAG_TILE_SHIFT bits of `flags`) so that the per-warp observation loop gets shorter
  const int ts = (int)((flags >> CZ_FLAG_TILE_SHIFT) & 7u), TS = 1 << ts;
  const int n_tiles = (n_envs + TS - 1) >> ts;
  const int warps_total = gridDim.x * CZ_WARPS_PER_BLOCK;
  const size_t N = (size_t)ld;
  const uint32_t* misc = state + (size_t)(D + A) * N;
  uint32_t* misc_out = state_out + (size_t)(D + A) * N;  // == misc unless the step is pipelined (ping-pong state)

  for (int tile = blockIdx.x * CZ_WARPS_PER_BLOCK + warp; tile < n_tiles; tile += warps_total) {
    const int env = (tile << ts) + lane;
    const bool valid = lane < TS && env < n_envs;
    EnvRegs e;
    e.o = ws->obj + lane;
    e.ag = ws->ag + lane;
    e.st = st;
    e.err = 0;
    e.sbits = 0; e.variant = 0;
    bool write_obs = valid;
    if (valid) {
      // ---- phase 1: state -> shared columns (coalesced: consecutive lanes, consecutive words);
      // every word of the environment is in flight at once (LDGSTS + plain loads), one wait
      for (int s = 0; s < D; ++s) cz_cp_async4(e.o + s * OSTRIDE, state + (size_t)s * N + env);
      for (int i = 0; i < A; ++i) cz_cp_async4(e.ag + i * OSTRIDE, state + (size_t)(D + i) * N + env);
      e.sbits = misc[(size_t)CZ_ROW_SBITS * N + env];
      e.tinfo = misc[(size_t)CZ_ROW_TINFO * N + env];
      e.marks = misc[(size_t)CZ_ROW_MARKS * N + env];
      e.variant = misc[(size_t)CZ_ROW_VARIANT * N + env];
      e.rids = misc[(size_t)CZ_ROW_RECIPES * N + env];
      e.episode = misc[(size_t)CZ_ROW_EPISODE * N + env];
      uint32_t act = 0;
      if (MODE == MODE_STEP)
        for (int i = 0; i < A; ++i) act |= (uint32_t)actions[(size_t)env * A + i] << (8 * i);
      cz_cp_async_wait_all();

      bool do_reset = false;
      int layout = 0;
      if (MODE == MODE_RESET) {
        do_reset = mask == nullptr || mask[env] != 0;
        write_obs = do_reset;
        if (do_reset) {
          layout = layout_ids[env];
          if ((unsigned)layout >= (unsigned)T.P) {  // a direct C caller passed an id outside the pool: clamp and flag
            layout = 0;
            e.err |= CZ_ERR_BAD_ID;
          }
          uint32_t rids = 0;
          for (int r = 0; r < T.R; ++r) {
            uint32_t id = recipe_ids ? recipe_ids[(size_t)env * T.R + r] : __ldg(T.default_recipes + r);
            if (id >= (uint32_t)T.B) {
              id = 0;
              e.err |= CZ_ERR_BAD_ID;
            }
            rids |= id << (8 * r);
          }
          e.rids = rids;
        }
      } else if (MODE == MODE_STEP) {
        if ((flags & CZ_STEP_AUTO_RESET) && (e.tinfo & TI_DONE)) {
          do_reset = true;
          layout = cz_pick_layout(T.layout_cum, T.P, cz_mix(seed, (uint64_t)(env_offset + env), (uint64_t)e.episode));
        }
      }

      if (do_reset) {
        // ---- CookingEnvironment.reset (cooking_env.py:178-210): pooled layout -> state
        const uint32_t* src = T.pool + (size_t)layout * T.rows;
        for (int s = 0; s < D; ++s) e.o[s * OSTRIDE] = __ldg(src + s);
        for (int i = 0; i < A; ++i) e.ag[i * OSTRIDE] = __ldg(src + D + i);
        e.sbits = __ldg(src + D + A + CZ_ROW_SBITS);
        e.tinfo = __ldg(src + D + A + CZ_ROW_TINFO);
        e.variant = __ldg(src + D + A + CZ_ROW_VARIANT);
        e.episode += 1;
        uint32_t marks = 0;
#pragma unroll 1
        for (int r = 0; r < T.R; ++r) marks |= cz_recipe_marks<FAST>(T, e, (e.rids >> (8 * r)) & 255u) << (8 * r);
        e.marks = marks;
        if (MODE == MODE_STEP) {
          for (int i = 0; i < A; ++i) {
            reward[(size_t)env * A + i] = 0.0;
            term[(size_t)env * A + i] = 0;
            trunc[(size_t)env * A + i] = 0;
          }
        }
      } else if (MODE == MODE_STEP) {
        // ---- phase 2: one accumulated_step per lane
        cz_step_env<FAST, NA>(T, e, act, reward + (size_t)env * A, term + (size_t)env * A, trunc + (size_t)env * A, seed,
                              (uint64_t)(env_offset + env));
      }

      // ---- phase 3: shared columns -> state
      if (MODE != MODE_OBSERVE && (MODE == MODE_STEP || do_reset)) {
        for (int s = 0; s < D; ++s) state_out[(size_t)s * N + env] = e.o[s * OSTRIDE];
        for (int i = 0; i < A; ++i) state_out[(size_t)(D + i) * N + env] = e.ag[i * OSTRIDE];
        misc_out[(size_t)CZ_ROW_SBITS * N + env] = e.sbits;
        misc_out[(size_t)CZ_ROW_TINFO * N + env] = e.tinfo;
        misc_out[(size_t)CZ_ROW_MARKS * N + env] = e.marks;
        misc_out[(size_t)CZ_ROW_VARIANT * N + env] = e.variant;
        misc_out[(size_t)CZ_ROW_RECIPES * N + env] = e.rids;
        misc_out[(size_t)CZ_ROW_EPISODE * N + env] = e.episode;
        if (errflags && e.err) errflags[env] |= e.err;
      }
    }
    ws->sbits[lane] = e.sbits;
    ws->variant[lane] = e.variant;
    ws->wobs[lane] = write_obs ? 1u : 0u;
    __syncwarp();

    if (OBS == OBS_NONE) continue;  // pipelined step: observations come from the observe kernel on the other stream
    // ---- phase 4: observation rows of the tile, one environment (A rows) at a time, whole warp
    // Its invariants are derived here, from an opaque copy of the lane id, so that they are not
    // hoisted above the dynamics (where they would be spilled: registers are capped for 28 warps/SM).
    int lane_o = lane;
    asm volatile("" : "+r"(lane_o));
    const int n_here = min(TS, n_envs - (tile << ts));
    double* genv = obs + ((size_t)tile << ts) * A * T.L;
    const size_t env_doubles = (size_t)A * T.L;
    const int tab2 = T.tab_len >> 1, L2 = T.L >> 1;
    const uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(stage);
    const size_t row_gbytes = (size_t)T.L * 8;
    const uint32_t r0_bytes = (uint32_t)T.ranges[0][1] * 8;
    const size_t r0_goff = (size_t)T.ranges[0][0] * 8;
    const uint32_t r0_soff = (uint32_t)(T.ranges[0][0] - T.stage_lo) * 8;
    if constexpr (FAST) {
      cz_obs_phase_fast<NA, OBS>(T, st, ws, sxl, syl, stage, stage_s, row_stride, (uint32_t)row_bytes, genv, n_here, lane_o, tab2, L2,
                            row_gbytes, r0_bytes, r0_goff, r0_soff);
      __syncwarp();
      continue;
    } else {
    const LaneSlot ls = cz_lane_slot(T, lane_o, 0, lane_o);
#pragma unroll 1
    for (int le = 0; le < n_here; ++le, genv += env_doubles) {
      if (!ws->wobs[le]) continue;
      const uint32_t sb = ws->sbits[le], var = ws->variant[le];
      const double2* tab = reinterpret_cast<const double2*>(T.obs_table) + (size_t)var * 64 * tab2 + lane;
      uint32_t xy = 0, fb = 0;
      if (ls.off >= 0) cz_slot_state<false>(T, st, ls, ws->obj, ws->ag, sb, var, le, xy, fb);
      if (OBS == OBS_TMA) {
        // the bulk stores of the previous environment must have finished reading the staging rows
        if (lane == 0) cz_bulk_wait_read<0>();
        __syncwarp();
      }
      double* row = stage;
      double2* g2 = reinterpret_cast<double2*>(genv);
#pragma unroll 1
      for (int a = 0; a < A; ++a, row += row_stride, g2 += L2) {
        const uint32_t me = ws->ag[a * OSTRIDE + le];
        const double2* src = tab + (me & 63u) * tab2;
        double2 v0, v1;
        if (ls.t0 >= 0) v0 = __ldg(src);
        if (ls.t1 >= 0) v1 = __ldg(src + 32);
        // one lane per slot, as many passes as it takes
        if (ls.off >= 0)
          cz_slot_store(ls, xy, fb, me & 7u, (me >> 3) & 7u, ls.kind == 2 && (int)ls.idx == a, sxl, syl, row);
        for (int q = lane + 32; q < T.n_comp; q += 32) {
          const LaneSlot l2 = cz_lane_slot(T, q, 0, lane);
          uint32_t xy2, fb2;
          cz_slot_state<false>(T, st, l2, ws->obj, ws->ag, sb, var, le, xy2, fb2);
          cz_slot_store(l2, xy2, fb2, me & 7u, (me >> 3) & 7u, l2.kind == 2 && (int)l2.idx == a, sxl, syl, row);
        }
        if (ls.t0 >= 0) g2[ls.t0] = v0;
        if (ls.t1 >= 0) g2[ls.t1] = v1;
        for (int k = lane + 64; k < tab2; k += 32) {  // table rows longer than 64 double2
          const int n0 = T.segs[0][1] >> 1;
          g2[k < n0 ? (T.segs[0][0] >> 1) + k : (T.segs[1][0] >> 1) + k - n0] = __ldg(src - lane + k);
        }
      }
      if (OBS == OBS_TMA) {
        cz_fence_async_smem();  // generic-proxy writes -> visible to the async proxy
        __syncwarp();
        if (lane == 0) {
          // one elected lane hands the computed range(s) of the A rows to the TMA engine
          char* gp = reinterpret_cast<char*>(genv) + r0_goff;
          uint32_t sp = stage_s + r0_soff;
#pragma unroll 1
          for (int a = 0; a < A; ++a, gp += row_gbytes, sp += (uint32_t)row_bytes) {
            cz_bulk_store_s(gp, sp, r0_bytes);
            for (int r = 1; r < T.n_ranges; ++r)
              cz_bulk_store_s(gp + (T.ranges[r][0] - T.ranges[0][0]) * 8, sp + (T.ranges[r][0] - T.ranges[0][0]) * 8,
                              (uint32_t)T.ranges[r][1] * 8);
          }
          cz_bulk_commit();
        }
      } else {
        __syncwarp();
        for (int a = 0; a < A; ++a) {
          for (int r = 0; r < T.n_ranges; ++r) {
            const double* srow = stage + a * row_stride + (T.ranges[r][0] - T.stage_lo);
            double* g = genv + (size_t)a * T.L + T.ranges[r][0];
            if ((T.L & 1) == 0) {  // rows and ranges are 16-byte aligned: 128-bit coalesced stores
              for (int k = lane; k < (T.ranges[r][1] >> 1); k += 32)
                reinterpret_cast<double2*>(g)[k] = reinterpret_cast<const double2*>(srow)[k];
            } else {
              for (int k = lane; k < T.ranges[r][1]; k += 32) g[k] = srow[k];
            }
          }
        }
        __syncwarp();
      }
    }
    if (OBS == OBS_TMA) {
      if (lane == 0) cz_bulk_wait_read<0>();  // staging and columns are reused by the next tile
    }
    __syncwarp();
    }
  }
}

// =========================================================================================
// Environment-per-warp observation writer (specialised configurations): obs = f(state), ONE WARP PER
// ENVIRONMENT (its NA rows), eight environments per block, tens of thousands of short blocks.
// Used by the pipelined step: short blocks retire continuously, so the high-priority dynamics
// kernel of the next step finds free SM slots and overlaps with this kernel's stores instead of
// queueing behind a single wave of long-running blocks.  A lane owns one (observer, slot) pair and
// reads its slot's state word straight from L2 (the dynamics kernel has just written it); the warp
// zero-fills and fills its private staging rows, then streams the computed range and the table
// segments out with 128-bit stores.  No TMA, no proxy fence, no block-level barrier.
// =========================================================================================
#ifndef ENVS_WARPS
#define ENVS_WARPS 8
#endif
#ifndef CZ_ENVS_MIN_BLOCKS
#define CZ_ENVS_MIN_BLOCKS (64 / ENVS_WARPS)
#endif

// A static slot among the computed ones (live Switch / Block, world_objects.py:174,221): its record is the cell with
// the present bit, its one state flag comes from the SBITS word.  Shared by the warp-per-environment row writers.
__device__ __forceinline__ void cz_live_static(const CzDev& T, const uint32_t* __restrict__ state, size_t N, int env, int A,
                                               uint32_t var, uint32_t idx, uint32_t& rec, uint32_t& fb4) {
  const uint32_t cell = __ldg(T.static_cells + var * T.S + idx);
  rec = cell != 0xFFu ? (cell | O_PRESENT) : 0u;
  const uint32_t g = __ldg(T.grid + var * 64 + (rec & 63u));
  const uint32_t sbits = __ldg(state + (size_t)(T.D + A + CZ_ROW_SBITS) * N + env);
  fb4 = ((g & 15u) == ST_SWITCH ? (sbits >> (12 + (g >> 4))) : (sbits >> (16 + (g >> 4)))) & 1u;
}

// State words of one (observer, slot) pair: the slot's record (or cell | present for a static slot) and its feature bits.
struct PairRegs {
  uint32_t rec, me, static_fb;
};

template <int NA>
__device__ __forceinline__ PairRegs cz_pair_load(const CzDev& T, const uint32_t* __restrict__ state, size_t N, int env,
                                                 uint32_t var, const LaneSlot& ls) {
  PairRegs p;
  p.rec = 0;
  p.static_fb = 0;
  const bool is_agent = ls.kind == 2, is_static = ls.kind == 0;
  if (ls.off >= 0 && !is_static) p.rec = __ldg(state + (size_t)(is_agent ? T.D + ls.idx : ls.idx) * N + env);
  p.me = __ldg(state + (size_t)(T.D + ls.agent) * N + env);  // this pair's observer
  if (ls.off >= 0 && is_static) cz_live_static(T, state, N, env, NA, var, ls.idx, p.rec, p.static_fb);
  return p;
}

// [x, y, flags..., 1] of the pair into its staging row
__device__ __forceinline__ void cz_pair_store_at(const CzDev& T, const LaneSlot& ls, const PairRegs& p, double* span0);
__device__ __forceinline__ void cz_pair_store(const CzDev& T, const LaneSlot& ls, const PairRegs& p, double2* stage, int stage2) {
  cz_pair_store_at(T, ls, p, reinterpret_cast<double*>(stage + ls.agent * stage2));
}
// `span0`: where element stage_lo of the pair's row lives (staged span or whole staged row)
__device__ __forceinline__ void cz_pair_store_at(const CzDev& T, const LaneSlot& ls, const PairRegs& p, double* span0) {
  if (ls.off < 0) return;
  const bool is_agent = ls.kind == 2, is_static = ls.kind == 0;
  const uint32_t rec = p.rec, me = p.me;
  const bool present = is_agent || (rec & O_PRESENT);
  const uint32_t c = (rec >> 7) & 1u, m = (rec >> 8) & 1u;
  const uint32_t fb4 = is_static ? p.static_fb : (is_agent ? ((1u << A_ORI(rec)) >> 1) : (((c | m) ^ 1u) | c << 1 | m << 2));
  const uint32_t one = 1u << (ls.flen - 1);
  const uint32_t fb = present ? ((fb4 & (one - 1u)) | one) : 0u;
  const bool self = is_agent && (int)ls.idx == ls.agent;
  const int x = rec & 7u, y = (rec >> 3) & 7u;
  // (x - ax) / W from the host-divided table; the observer's own entry is x / W (cooking_env.py:364-368)
  double X = __ldg(T.xlut + (x - (self ? 0 : (int)(me & 7u)) + T.W - 1));
  double Y = __ldg(T.ylut + (y - (self ? 0 : (int)((me >> 3) & 7u)) + T.H - 1));
  if (!present) { X = 0.0; Y = 0.0; }
  double* out = span0 + ls.off;
  out[0] = X;
  out[1] = Y;
#pragma unroll
  for (int k = 0; k < 5; ++k)
    if (k < (int)ls.flen) *reinterpret_cast<uint2*>(out + 2 + k) = make_uint2(0u, (fb >> k & 1u) ? 0x3FF00000u : 0u);
}

#ifndef CZ_ENVS_TMA
#define CZ_ENVS_TMA 1  // computed range of the rows through cp.async.bulk: the same time alone and in place, but fewer issue slots
                       // taken from the background dynamics of the pipelined step (104.75 -> 102.74 us); 0: lane copies (A/B build)
#endif
// TWO = false: at most 32 (observer, slot) pairs, one per lane.  TWO = true: up to 64 pairs (3-4 agent kitchens),
// a lane owns pairs `lane` and `lane + 32`.
template <int NA, bool TWO>
__global__ void __launch_bounds__(32 * ENVS_WARPS, (TWO || NA >= 3) ? 5 : CZ_ENVS_MIN_BLOCKS)
cz_obs_envs_kernel(const __grid_constant__ CzDev T, const uint32_t* __restrict__ state, double* __restrict__ obs, int n_envs, int ld) {
  extern __shared__ __align__(16) unsigned char smem_rows[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int env = blockIdx.x * ENVS_WARPS + warp;
  if (env >= n_envs) return;
  const int D = T.D, tab2 = T.tab_len >> 1, L2 = T.L >> 1;
  const size_t N = (size_t)ld;  // columns of the state matrix (the launch may cover a column range of a larger batch)
  const int stage2 = (T.stage_len + 1) >> 1;  // double2 per staging row
  double2* stage = reinterpret_cast<double2*>(smem_rows) + (size_t)warp * NA * stage2;

  // this lane's (observer, slot) pair(s) and the state words they need
  const uint32_t var = __ldg(state + (size_t)(D + NA + CZ_ROW_VARIANT) * N + env);
  const LaneSlot ls = cz_lane_slot_packed(T, lane);
  const PairRegs p = cz_pair_load<NA>(T, state, N, env, var, ls);
  LaneSlot ls1;
  PairRegs p1;
  if constexpr (TWO) {
    ls1 = cz_lane_slot_packed(T, lane + 32);
    p1 = cz_pair_load<NA>(T, state, N, env, var, ls1);
  }
  const double2* tab = reinterpret_cast<const double2*>(T.obs_table) + (size_t)var * 64 * tab2 + lane;
  double2* g2 = reinterpret_cast<double2*>(obs + (size_t)env * NA * T.L);
  // never-occupied slots are zeros: clear the staging rows, then fill the live slots
  for (int k = lane; k < NA * stage2; k += 32) stage[k] = make_double2(0.0, 0.0);
  __syncwarp();
  cz_pair_store(T, ls, p, stage, stage2);
  if constexpr (TWO) cz_pair_store(T, ls1, p1, stage, stage2);
#if CZ_ENVS_TMA
  cz_fence_async_smem();  // generic-proxy writes -> visible to the async proxy
#endif
  __syncwarp();
  {
    const int n2 = T.ranges[0][1] >> 1, o2 = T.ranges[0][0] >> 1, s2 = (T.ranges[0][0] - T.stage_lo) >> 1;
#if CZ_ENVS_TMA
    if (lane == 0) {  // the computed range of the NA rows leaves through the TMA engine
#pragma unroll
      for (int a = 0; a < NA; ++a) cz_bulk_store_nocommit(g2 + a * L2 + o2, stage + a * stage2 + s2, (uint32_t)n2 * 16u);
      cz_bulk_commit();
    }
#else
#pragma unroll
    for (int a = 0; a < NA; ++a)
      for (int k = lane; k < n2; k += 32) cz_row_store(g2 + a * L2 + o2 + k, stage[a * stage2 + s2 + k]);
#endif
  }
  {  // table segments: all rows' loads first, then the stores
    double2 v0[NA], v1[NA];
#pragma unroll
    for (int a = 0; a < NA; ++a) {
      uint32_t cell;
      if constexpr (TWO) cell = __ldg(state + (size_t)(D + a) * N + env) & 63u;
      else cell = __shfl_sync(0xffffffffu, p.me, a * T.n_comp) & 63u;  // lane a*n_comp observes for agent a
      if (ls.t0 >= 0) v0[a] = __ldg(tab + cell * tab2);
      if (ls.t1 >= 0) v1[a] = __ldg(tab + cell * tab2 + 32);
    }
#pragma unroll
    for (int a = 0; a < NA; ++a) {
      if (ls.t0 >= 0) cz_row_store(g2 + a * L2 + ls.t0, v0[a]);
      if (ls.t1 >= 0) cz_row_store(g2 + a * L2 + ls.t1, v1[a]);
    }
  }
#if CZ_ENVS_TMA
  if (lane == 0) cz_bulk_wait_read<0>();  // the staging rows must outlive the bulk reads
#endif
}

// Single-agent batches: a row is only 2224 bytes, 4.3 sixteen-byte elements per lane, and the one-environment writer spends
// its life waiting for its loads (4.4 TB/s).  Here a warp builds the rows of TWO neighbouring environments whole in shared
// memory — table segments by cp.async (no registers), computed slots by the lanes, both environments' loads in flight
// together — and hands the 2 * L doubles to the TMA engine as one bulk store (the float32 pair writer, cz_obs32.cuh).
__device__ __forceinline__ void cz_cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}

__global__ void __launch_bounds__(32 * ENVS_WARPS, 6)
cz_obs_single_pair_kernel(const __grid_constant__ CzDev T, const uint32_t* __restrict__ state, double* __restrict__ obs, int n_envs,
                          int ld) {
  extern __shared__ __align__(16) unsigned char smem_rows[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int env0 = (blockIdx.x * ENVS_WARPS + warp) * 2;
  if (env0 >= n_envs) return;
  const bool two = env0 + 1 < n_envs;
  const int env1 = two ? env0 + 1 : env0;  // a lone last environment is built twice and written once
  const int D = T.D, tab2 = T.tab_len >> 1, L2 = T.L >> 1;
  const size_t N = (size_t)ld;
  double2* rows = reinterpret_cast<double2*>(smem_rows) + (size_t)warp * 2 * L2;

  const LaneSlot ls = cz_lane_slot_packed(T, lane);
  const uint32_t var0 = __ldg(state + (size_t)(D + 1 + CZ_ROW_VARIANT) * N + env0);
  const uint32_t var1 = __ldg(state + (size_t)(D + 1 + CZ_ROW_VARIANT) * N + env1);
  const PairRegs p0 = cz_pair_load<1>(T, state, N, env0, var0, ls);
  const PairRegs p1 = cz_pair_load<1>(T, state, N, env1, var1, ls);
  {  // table segments of both rows: lane 0 holds the observer
    const uint32_t c0 = __shfl_sync(0xffffffffu, p0.me, 0) & 63u, c1 = __shfl_sync(0xffffffffu, p1.me, 0) & 63u;
    const double2* tab0 = reinterpret_cast<const double2*>(T.obs_table) + ((size_t)var0 * 64 + c0) * tab2 + lane;
    const double2* tab1 = reinterpret_cast<const double2*>(T.obs_table) + ((size_t)var1 * 64 + c1) * tab2 + lane;
    if (ls.t0 >= 0) {
      cz_cp_async16(rows + ls.t0, tab0);
      cz_cp_async16(rows + L2 + ls.t0, tab1);
    }
    if (ls.t1 >= 0) {
      cz_cp_async16(rows + ls.t1, tab0 + 32);
      cz_cp_async16(rows + L2 + ls.t1, tab1 + 32);
    }
  }
  {  // never-occupied slots of the computed range are zeros
    const int n2 = T.ranges[0][1] >> 1, o2 = T.ranges[0][0] >> 1;
    for (int k = lane; k < n2; k += 32) {
      rows[o2 + k] = make_double2(0.0, 0.0);
      rows[L2 + o2 + k] = make_double2(0.0, 0.0);
    }
  }
  __syncwarp();
  cz_pair_store_at(T, ls, p0, reinterpret_cast<double*>(rows) + T.stage_lo);
  cz_pair_store_at(T, ls, p1, reinterpret_cast<double*>(rows + L2) + T.stage_lo);
  cz_cp_async_wait_all();
  cz_fence_async_smem();  // generic-proxy and cp.async writes -> visible to the async proxy
  __syncwarp();
  if (lane == 0) {
    cz_bulk_store_stream(obs + (size_t)env0 * T.L, rows, (uint32_t)((two ? 2 : 1) * T.L) * 8u);
    cz_bulk_commit();
    cz_bulk_wait_read<0>();  // the staged rows must outlive the read
  }
}

// Whole rows through the TMA engine (packed plans with at most 32 pairs, 2+ agents): one environment per warp, its NA rows
// staged whole in shared memory — table segments by cp.async (no registers), zeros and computed slots by the lanes — and ONE
// bulk store of NA * L doubles with the L2 evict_first hint (cz_bulk_store_stream).  Nothing else writes into the block's lines,
// which is what lets the hint work: 6.4-6.7 TB/s against 6.2 TB/s for the writer that mixes bulk and lane stores.
template <int NA, bool TWO>
__global__ void __launch_bounds__(32 * ENVS_WARPS, (TWO ? 3 : 6) * 8 / ENVS_WARPS)
cz_obs_whole_kernel(const __grid_constant__ CzDev T, const uint32_t* __restrict__ state, double* __restrict__ obs, int n_envs, int ld) {
  extern __shared__ __align__(16) unsigned char smem_rows[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int env = blockIdx.x * ENVS_WARPS + warp;
  if (env >= n_envs) return;
  const int D = T.D, tab2 = T.tab_len >> 1, L2 = T.L >> 1;
  const size_t N = (size_t)ld;
  double2* rows = reinterpret_cast<double2*>(smem_rows) + (size_t)warp * NA * L2;

  const LaneSlot ls = cz_lane_slot_packed(T, lane);
  const uint32_t var = __ldg(state + (size_t)(D + NA + CZ_ROW_VARIANT) * N + env);
  const PairRegs p = cz_pair_load<NA>(T, state, N, env, var, ls);
  LaneSlot ls1;
  PairRegs p1;
  if constexpr (TWO) {  // 33-64 (observer, slot) pairs: a lane owns pairs `lane` and `lane + 32`
    ls1 = cz_lane_slot_packed(T, lane + 32);
    p1 = cz_pair_load<NA>(T, state, N, env, var, ls1);
  }
  {
    const double2* tab = reinterpret_cast<const double2*>(T.obs_table) + (size_t)var * 64 * tab2 + lane;
#pragma unroll
    for (int a = 0; a < NA; ++a) {
      uint32_t cell;
      if constexpr (TWO) cell = __ldg(state + (size_t)(D + a) * N + env) & 63u;
      else cell = __shfl_sync(0xffffffffu, p.me, a * T.n_comp) & 63u;  // lane a * n_comp observes for agent a
      if (ls.t0 >= 0) cz_cp_async16(rows + a * L2 + ls.t0, tab + cell * tab2);
      if (ls.t1 >= 0) cz_cp_async16(rows + a * L2 + ls.t1, tab + cell * tab2 + 32);
    }
  }
  {  // never-occupied slots of the computed range are zeros
    const int n2 = T.ranges[0][1] >> 1, o2 = T.ranges[0][0] >> 1;
#pragma unroll
    for (int a = 0; a < NA; ++a)
      for (int k = lane; k < n2; k += 32) rows[a * L2 + o2 + k] = make_double2(0.0, 0.0);
  }
  __syncwarp();
  cz_pair_store_at(T, ls, p, reinterpret_cast<double*>(rows + ls.agent * L2) + T.stage_lo);
  if constexpr (TWO) cz_pair_store_at(T, ls1, p1, reinterpret_cast<double*>(rows + ls1.agent * L2) + T.stage_lo);
  cz_cp_async_wait_all();
  cz_fence_async_smem();  // generic-proxy and cp.async writes -> visible to the async proxy
  __syncwarp();
  if (lane == 0) {
    cz_bulk_store_stream(obs + (size_t)env * NA * T.L, rows, (uint32_t)(NA * T.L) * 8u);
    cz_bulk_commit();
    cz_bulk_wait_read<0>();  // the staged rows must outlive the read
  }
}

// The same writer for ANY observation plan (tables outside the packed class: more than 64 (observer, slot) pairs, table runs
// longer than 128 doubles, several computed ranges, odd row lengths, more than 16 variants): one warp per environment, loops
// where the packed writer has one or two elements per lane, tables read from global memory.  The staging rows hold the whole
// span of the computed ranges; with an even row length everything moves as 16-byte elements, otherwise as doubles.
template <bool EVEN>
__global__ void __launch_bounds__(32 * ENVS_WARPS, 8)  // 32 registers: a full SM of warps is worth more than the spills (0.73 vs 0.64 / 0.47 of roofline at 6 / 4 blocks)
cz_obs_any_kernel(const __grid_constant__ CzDev T, const uint32_t* __restrict__ state, double* __restrict__ obs, int n_envs, int ld,
                  int warps_per_block) {
  extern __shared__ __align__(16) unsigned char smem_any[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int env = blockIdx.x * warps_per_block + warp;
  if (warp >= warps_per_block || env >= n_envs) return;
  const int A = T.A, D = T.D, L = T.L;
  const size_t N = (size_t)ld;
  const int span = (T.stage_len + 1) & ~1;  // doubles per staging row (even: rows stay 16-byte aligned)
  double* stage = reinterpret_cast<double*>(smem_any) + (size_t)warp * A * span;
  const uint32_t* misc = state + (size_t)(D + A) * N;
  const uint32_t var = __ldg(misc + (size_t)CZ_ROW_VARIANT * N + env);
  const uint32_t sbits = __ldg(misc + (size_t)CZ_ROW_SBITS * N + env);
  for (int k = lane; k < (A * span) >> 1; k += 32)  // never-occupied slots are zeros (span is even: 16-byte elements)
    reinterpret_cast<double2*>(stage)[k] = make_double2(0.0, 0.0);
  __syncwarp();
  // computed slots: a lane takes (observer, slot) pairs lane, lane + 32, ... (pair p = observer * n_comp + slot)
  const int n_pairs = A * T.n_comp;
  for (int pr = lane; pr < n_pairs; pr += 32) {
    const int a = (pr >= T.n_comp) + (pr >= 2 * T.n_comp) + (pr >= 3 * T.n_comp);  // A <= 4: no division
    const int q = pr - a * T.n_comp;
    const uint32_t d = __ldg(T.comp_slots + q);
    const int off = (int)(d & 0xFFFu) - T.stage_lo;
    const uint32_t flen = (d >> 12) & 7u, kind = (d >> 15) & 3u, idx = (d >> 17) & 255u;
    uint32_t rec = 0, fb4 = 0;
    bool present;
    if (kind != 0u) {
      const bool is_agent = kind == 2u;
      const bool exists = !is_agent || (int)idx < A;
      rec = exists ? __ldg(state + (size_t)(is_agent ? D + idx : idx) * N + env) : 0u;
      present = is_agent ? exists : (rec & O_PRESENT) != 0;
      const uint32_t c = (rec >> 7) & 1u, m = (rec >> 8) & 1u;
      fb4 = is_agent ? ((1u << A_ORI(rec)) >> 1) : (((c | m) ^ 1u) | c << 1 | m << 2);
    } else {  // live Switch / Block (world_objects.py:174,221)
      const uint32_t cell = __ldg(T.static_cells + var * T.S + idx);
      present = cell != 0xFFu;
      rec = present ? cell : 0u;
      const uint32_t g = __ldg(T.grid + var * 64 + rec);
      fb4 = ((g & 15u) == ST_SWITCH ? (sbits >> (12 + (g >> 4))) : (sbits >> (16 + (g >> 4)))) & 1u;
    }
    const uint32_t one = 1u << (flen - 1);
    const uint32_t fb = present ? ((fb4 & (one - 1u)) | one) : 0u;
    const int x = rec & 7u, y = (rec >> 3) & 7u;
    const uint32_t me = __ldg(state + (size_t)(D + a) * N + env);
    const bool self = kind == 2u && (int)idx == a;  // the observer's own entry is x / W, y / H (cooking_env.py:364-368)
    double X = __ldg(T.xlut + (x - (self ? 0 : (int)(me & 7u)) + T.W - 1));
    double Y = __ldg(T.ylut + (y - (self ? 0 : (int)((me >> 3) & 7u)) + T.H - 1));
    if (!present) { X = 0.0; Y = 0.0; }
    double* out = stage + a * span + off;
    out[0] = X;
    out[1] = Y;
#pragma unroll
    for (uint32_t k = 0; k < 5; ++k)
      if (k < flen) *reinterpret_cast<uint2*>(out + 2 + k) = make_uint2(0u, (fb >> k & 1u) ? 0x3FF00000u : 0u);
  }
  if (EVEN) cz_fence_async_smem();  // generic-proxy writes -> visible to the async proxy
  __syncwarp();
  double* genv = obs + (size_t)env * A * L;
  bool bulk = false;
  for (int a = 0; a < A; ++a) {
    double* grow = genv + (size_t)a * L;
    const double* srow = stage + a * span;
    for (int r = 0; r < T.n_ranges; ++r) {  // computed ranges: staging -> row
      const int o = T.ranges[r][0], n = T.ranges[r][1], so = o - T.stage_lo;
      if (EVEN && !((o | n | so) & 1)) {  // 16-byte aligned on both sides, a multiple of 16 bytes: one bulk store (TMA engine)
        if (lane == 0) cz_bulk_store_nocommit(grow + o, srow + so, (uint32_t)n * 8u);
        bulk = true;
      } else {
        for (int k = lane; k < n; k += 32) grow[o + k] = srow[so + k];
      }
    }
    const uint32_t cell = __ldg(state + (size_t)(D + a) * N + env) & 63u;
    const double* tab = T.obs_table + ((size_t)var * 64 + cell) * T.tab_len;
    for (int sg = 0; sg < T.n_segs; ++sg) {  // table segments (even offsets and lengths by construction): table -> row
      const int o = T.segs[sg][0], n = T.segs[sg][1], to = T.segs[sg][2];
      if (EVEN) {
        for (int k = lane; k < (n >> 1); k += 32)
          reinterpret_cast<double2*>(grow + o)[k] = __ldg(reinterpret_cast<const double2*>(tab + to) + k);
      } else {
        for (int k = lane; k < n; k += 32) grow[o + k] = __ldg(tab + to + k);
      }
    }
  }
  if (bulk && lane == 0) {
    cz_bulk_commit();
    cz_bulk_wait_read<0>();  // the staging rows must outlive the bulk reads
  }
}

// The any-plan writer with WHOLE rows staged (A * L even, so that an environment's block is 16-byte aligned): table
// segments by cp.async into their place in the staged rows, zeros over the computed ranges, computed slots by the lanes, and
// one bulk store of the environment's A * L doubles with the L2 evict_first hint — the structure of cz_obs_whole_kernel
// with loops where that kernel has one element per lane.
__device__ __forceinline__ void cz_cp_async8d(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}

__global__ void __launch_bounds__(32 * ENVS_WARPS, 5)
cz_obs_any_whole_kernel(const __grid_constant__ CzDev T, const uint32_t* __restrict__ state, double* __restrict__ obs, int n_envs,
                        int ld, int warps_per_block) {
  extern __shared__ __align__(16) unsigned char smem_any[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int env = blockIdx.x * warps_per_block + warp;
  if (warp >= warps_per_block || env >= n_envs) return;
  const int A = T.A, D = T.D, L = T.L;
  const size_t N = (size_t)ld;
  double* rows = reinterpret_cast<double*>(smem_any) + (size_t)warp * A * L;  // A * L is even: every warp's block is 16-byte aligned
  const uint32_t* misc = state + (size_t)(D + A) * N;
  const uint32_t var = __ldg(misc + (size_t)CZ_ROW_VARIANT * N + env);
  const uint32_t sbits = __ldg(misc + (size_t)CZ_ROW_SBITS * N + env);
  const bool even = (L & 1) == 0;
  for (int a = 0; a < A; ++a) {
    double* srow = rows + a * L;
    const uint32_t cell = __ldg(state + (size_t)(D + a) * N + env) & 63u;
    const double* tab = T.obs_table + ((size_t)var * 64 + cell) * T.tab_len;
    for (int sg = 0; sg < T.n_segs; ++sg) {  // table segments: table -> their place in the staged row, no registers
      const int o = T.segs[sg][0], n = T.segs[sg][1], to = T.segs[sg][2];
      if (even && !((o | n | to) & 1)) {
        for (int k = lane; k < (n >> 1); k += 32) cz_cp_async16(srow + o + 2 * k, tab + to + 2 * k);
      } else {
        for (int k = lane; k < n; k += 32) cz_cp_async8d(srow + o + k, tab + to + k);
      }
    }
    for (int r = 0; r < T.n_ranges; ++r) {  // never-occupied slots of the computed ranges are zeros
      const int o = T.ranges[r][0], n = T.ranges[r][1];
      for (int k = lane; k < n; k += 32) srow[o + k] = 0.0;
    }
  }
  __syncwarp();
  // computed slots: a lane takes (observer, slot) pairs lane, lane + 32, ... (pair p = observer * n_comp + slot)
  const int n_pairs = A * T.n_comp;
  for (int pr = lane; pr < n_pairs; pr += 32) {
    const int a = (pr >= T.n_comp) + (pr >= 2 * T.n_comp) + (pr >= 3 * T.n_comp);  // A <= 4: no division
    const int q = pr - a * T.n_comp;
    const uint32_t d = __ldg(T.comp_slots + q);
    const int off = (int)(d & 0xFFFu);
    const uint32_t flen = (d >> 12) & 7u, kind = (d >> 15) & 3u, idx = (d >> 17) & 255u;
    uint32_t rec = 0, fb4 = 0;
    bool present;
    if (kind != 0u) {
      const bool is_agent = kind == 2u;
      const bool exists = !is_agent || (int)idx < A;
      rec = exists ? __ldg(state + (size_t)(is_agent ? D + idx : idx) * N + env) : 0u;
      present = is_agent ? exists : (rec & O_PRESENT) != 0;
      const uint32_t c = (rec >> 7) & 1u, m = (rec >> 8) & 1u;
      fb4 = is_agent ? ((1u << A_ORI(rec)) >> 1) : (((c | m) ^ 1u) | c << 1 | m << 2);
    } else {  // live Switch / Block (world_objects.py:174,221)
      const uint32_t cell = __ldg(T.static_cells + var * T.S + idx);
      present = cell != 0xFFu;
      rec = present ? cell : 0u;
      const uint32_t g = __ldg(T.grid + var * 64 + rec);
      fb4 = ((g & 15u) == ST_SWITCH ? (sbits >> (12 + (g >> 4))) : (sbits >> (16 + (g >> 4)))) & 1u;
    }
    const uint32_t one = 1u << (flen - 1);
    const uint32_t fb = present ? ((fb4 & (one - 1u)) | one) : 0u;
    const int x = rec & 7u, y = (rec >> 3) & 7u;
    const uint32_t me = __ldg(state + (size_t)(D + a) * N + env);
    const bool self = kind == 2u && (int)idx == a;  // the observer's own entry is x / W, y / H (cooking_env.py:364-368)
    double X = __ldg(T.xlut + (x - (self ? 0 : (int)(me & 7u)) + T.W - 1));
    double Y = __ldg(T.ylut + (y - (self ? 0 : (int)((me >> 3) & 7u)) + T.H - 1));
    if (!present) { X = 0.0; Y = 0.0; }
    double* out = rows + a * L + off;
    out[0] = X;
    out[1] = Y;
#pragma unroll
    for (uint32_t k = 0; k < 5; ++k)
      if (k < flen) *reinterpret_cast<uint2*>(out + 2 + k) = make_uint2(0u, (fb >> k & 1u) ? 0x3FF00000u : 0u);
  }
  cz_cp_async_wait_all();
  cz_fence_async_smem();  // generic-proxy and cp.async writes -> visible to the async proxy
  __syncwarp();
  if (lane == 0) {
    cz_bulk_store_stream(obs + (size_t)env * A * L, rows, (uint32_t)(A * L) * 8u);
    cz_bulk_commit();
    cz_bulk_wait_read<0>();  // the staged rows must outlive the read
  }
}

#include "cz_grid.cuh"
#include "cz_stats.cuh"

// =========================================================================================
// Host side: tables object and the C ABI
// =========================================================================================
static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

static int cz_fail(int code, const char* fmt, const char* detail) {
  snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}
#define CZ_CUDA(call)                                                              \
  do {                                                                             \
    cudaError_t _e = (call);                                                       \
    if (_e != cudaSuccess) return cz_fail(CZ_ECUDA, #call ": %s", cudaGetErrorString(_e)); \
  } while (0)

struct cz_tables {
  CzDev dev;
  int device;
  int obs_path;
  int simple;
  int simple2;
  int two_kernel_min_envs;  // in-place step of at least this many environments: dynamics kernel, then the row-writer kernel
  int warp_max_envs;        // single in-place step of at most this many environments: warp-per-environment kernel (cz_warp.cuh)
  int warp_k_max_envs;      // k_steps > 1 with at most this many environments: one persistent launch of that kernel
  int warp_group;           // lanes per environment in that kernel: 16 (two environments per warp) or 32
  uint64_t* h_layout_cum;   // host copy of the weighted pool's thresholds (cz_layout_index), or nullptr
  uint8_t* d_rand;          // scratch for device-generated actions outside the warp kernel
  int rand_envs;
  void* d_keep;             // scratch rows of one step of a KEEP_ALL call whose per-step block is not 16-byte aligned
  size_t keep_bytes;
  int num_sms;
  void* allocs[32];
  int n_allocs;
  // scratch for cz_step_host
  uint8_t* d_actions; double* d_obs; double* d_reward; uint8_t* d_term; uint8_t* d_trunc;
  int scratch_envs;
  // pipelined step: dynamics on a high-priority stream, observations on a second one, ping-pong state
  cudaStream_t pipe_dyn, pipe_obs;
  cudaEvent_t ev_user, ev_dyn, ev_obs[4], ev_chunk[8], ev_pol_in, ev_pol_out;
  int policy_on_dyn;        // cz_policy_act of a running pipeline launches on the dynamics stream (CZ_POLICY_ON_DYN=0: caller's stream)
  int fast_dyn;             // dynamics on the specialised (shared-memory table) kernels: V <= 16 variants and B <= 16 recipes,
                            // whatever the observation plan looks like
  int whole_rows;           // A >= 2 packed plans: whole rows staged, one bulk store per environment (bit 0: in place, bit 1: pipelined, bit 2: also the 33-64 pair plans, bit 3: the any-plan writer; CZ_WHOLE_ROWS)
  int single_pair;          // float64 rows of large single-agent batches: two environments per warp (CZ_SINGLE_PAIR=0: one)
  int obs32_pair;           // float32 rows of large batches: two environments per warp (CZ_OBS32_PAIR=0: one)
  int any_writer;           // generic tables, large in-place batches: dynamics kernel + any-plan row writer (CZ_ANY_WRITER=0: fused kernel)
  int host_chunks;          // cz_step_host: column ranges whose device->host copies overlap the stepping of the next range
  int split;                // in-place step of a large batch: column ranges whose dynamics run under the previous range's rows
  int pipe_ready, pipe_cur, pipe_obs_pending[4];
  int pipe_buffers;         // state matrices of the pipelined step's ring (2..4, cz_pipeline_config)
  int pipe_steps;           // pipelined steps enqueued since the last cz_pipeline_reset (0: the internal streams hold nothing to wait for)
  int pipe_dyn_blocks;   // blocks per SM the dynamics kernel of the pipelined step is launched with (0 = no cap): a small grid that
                         // loops over its tiles runs in the background of the row writer instead of displacing it
  size_t smem_optin;
  CzGridDev grid;           // the grid observation writer's constants (cz_grid.cuh)
  CzStatsDev stats;         // episode statistics buffers of cz_stats_attach (stats.n == 0: none attached)
};

template <typename Tp>
static int upload(cz_tables* t, const Tp* host, size_t count, const Tp** out) {
  *out = nullptr;
  if (count == 0) count = 1;
  void* d = nullptr;
  CZ_CUDA(cudaMalloc(&d, count * sizeof(Tp)));
  t->allocs[t->n_allocs++] = d;
  if (host) CZ_CUDA(cudaMemcpy(d, host, count * sizeof(Tp), cudaMemcpyHostToDevice));
  else CZ_CUDA(cudaMemset(d, 0, count * sizeof(Tp)));
  *out = (const Tp*)d;
  return CZ_OK;
}

static size_t cz_smem_bytes(const CzDev& T) {
  size_t row_bytes = ((size_t)T.stage_len * 8 + 15) & ~(size_t)15;
  return ((cz_block_smem_head(T.V) + cz_warp_words(T.D, T.A) * 4 * CZ_WARPS_PER_BLOCK + 15) & ~(size_t)15) +
         (size_t)CZ_WARPS_PER_BLOCK * CZ_STAGE_SETS * T.A * row_bytes;
}

#include "cz_obs32.cuh"
#include "cz_warp.cuh"

extern "C" int cz_abi_version(void) { return CZ_ABI_VERSION; }
extern "C" const char* cz_last_error(void) { return g_err; }
extern "C" uint64_t cz_launch_count(void) { return g_launches.load(); }

extern "C" uint64_t cz_layout_draw(uint64_t seed, uint64_t env, uint64_t episode) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (env + 1) + 0xD1B54A32D192ED03ull * (episode + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

extern "C" int cz_layout_index(const cz_tables* t, uint64_t seed, uint64_t env, uint64_t episode) {
  if (!t) return cz_fail(CZ_EINVAL, "%s", "null argument");
  return cz_pick_layout(t->h_layout_cum, t->dev.P, cz_layout_draw(seed, env, episode));
}

extern "C" double cz_spawn_uniform(uint64_t seed, uint64_t env, uint64_t episode, uint64_t t, uint64_t c) {
  return cz_uniform(seed, env, episode, t, c);
}

extern "C" int cz_tables_create(const cz_table_desc* d, int device, cz_tables** out) {
  if (!d || !out) return cz_fail(CZ_EINVAL, "%s", "null argument");
  *out = nullptr;
  if (d->abi_version != CZ_ABI_VERSION) return cz_fail(CZ_EINVAL, "%s", "cz_table_desc.abi_version mismatch");
  if (d->width < 1 || d->width > 8 || d->height < 1 || d->height > 8) return cz_fail(CZ_ELIMIT, "%s", "level larger than 8x8");
  if (d->num_agents < 1 || d->num_agents > CZ_MAX_AGENTS) return cz_fail(CZ_ELIMIT, "%s", "num_agents out of range");
  if (d->num_recipes < 1 || d->num_recipes > CZ_MAX_RECIPES) return cz_fail(CZ_ELIMIT, "%s", "num_recipes out of range");
  if (d->num_dyn_slots < 1 || d->num_dyn_slots > CZ_MAX_DYN) return cz_fail(CZ_ELIMIT, "%s", "num_dyn_slots out of range");
  if (d->num_types < 1 || d->num_types > CZ_MAX_TYPES) return cz_fail(CZ_ELIMIT, "%s", "num_types out of range");
  if (d->num_static_slots < 0 || d->num_static_slots > CZ_MAX_STATIC_SLOTS) return cz_fail(CZ_ELIMIT, "%s", "num_static_slots out of range");
  if (d->obs_len < 1 || d->obs_len > 4095) return cz_fail(CZ_ELIMIT, "%s", "obs_len out of range");
  if (d->num_variants < 1 || d->num_layouts < 1 || d->num_book < 1 || d->num_book > 255) return cz_fail(CZ_EINVAL, "%s", "empty tables");
  if (d->max_steps < 1 || d->max_steps >= (1 << 20)) return cz_fail(CZ_ELIMIT, "%s", "max_steps out of range");
  if (d->grace_period < 0 || d->grace_period > 65535) return cz_fail(CZ_ELIMIT, "%s", "grace_period out of range");
  CZ_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  CZ_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return cz_fail(CZ_ECUDA, "%s", "libcz_b200 is built for sm_100a (B200) only");
  cz_tables* t = new (std::nothrow) cz_tables();
  if (!t) return cz_fail(CZ_EINVAL, "%s", "out of host memory");
  memset(t, 0, sizeof(*t));
  t->device = device;
  t->num_sms = prop.multiProcessorCount;
  t->smem_optin = prop.sharedMemPerBlockOptin;
  {
    const char* pb = getenv("CZ_PIPE_DYN_BLOCKS");
    t->pipe_dyn_blocks = pb ? atoi(pb) : 0;
    t->pipe_buffers = 2;
  }
  const char* p = getenv("CZ_OBS_PATH");
  t->obs_path = (p && !strcmp(p, "stg")) ? OBS_STG : OBS_TMA;
  if (d->obs_len & 1) t->obs_path = OBS_STG;  // bulk copies need 16-byte rows
  static_assert(sizeof(VarTabs) % 16 == 0 && sizeof(BlockSmem) % 8 == 0, "block image is copied in 16-byte units");
  CzDev& T = t->dev;
  T.W = d->width; T.H = d->height; T.A = d->num_agents; T.R = d->num_recipes; T.D = d->num_dyn_slots;
  T.S = d->num_static_slots; T.T = d->num_types; T.L = d->obs_len;
  T.n_comp = d->num_comp_slots; T.n_segs = d->num_obs_segs; T.n_ranges = d->num_obs_ranges; T.tab_len = d->obs_table_len;
  if (T.n_segs < 0 || T.n_segs > 2 || T.n_ranges < 0 || T.n_ranges > 3 || T.n_comp < 0 || T.tab_len < 0)
    { delete t; return cz_fail(CZ_EINVAL, "%s", "bad observation plan"); }
  for (int i = 0; i < 2; ++i) for (int j = 0; j < 3; ++j) T.segs[i][j] = d->obs_segs[i][j];
  for (int i = 0; i < 3; ++i) for (int j = 0; j < 2; ++j) T.ranges[i][j] = d->obs_ranges[i][j];
  T.stage_lo = 0; T.stage_len = 2;
  if (T.n_ranges > 0) {
    T.stage_lo = T.ranges[0][0];
    T.stage_len = T.ranges[T.n_ranges - 1][0] + T.ranges[T.n_ranges - 1][1] - T.stage_lo;
  }
  if ((T.L & 1) && T.n_segs > 0) { delete t; return cz_fail(CZ_EINVAL, "%s", "table segments need an even obs_len"); }
  T.V = d->num_variants; T.P = d->num_layouts; T.B = d->num_book; T.max_steps = d->max_steps;
  T.scheme = d->action_scheme == 1 ? 1 : 3;
  T.end_all = d->end_all; T.grace = d->grace_period; T.n_switches = d->num_switches; T.n_blocks = d->num_blocks;
  T.rows = T.D + T.A + CZ_NUM_MISC_ROWS;
  T.r_node = d->reward_node; T.r_recipe = d->reward_recipe; T.r_penalty = d->reward_penalty; T.r_time = d->reward_time;
  T.respawn = d->respawn_rate; T.despawn = d->despawn_rate;
  int rc = CZ_OK;
#define UP(field, src, count) if (rc == CZ_OK) rc = upload(t, src, (size_t)(count), &T.field)
  UP(xlut, d->xlut, 2 * T.W - 1);
  UP(ylut, d->ylut, 2 * T.H - 1);
  UP(grid, d->grid, (size_t)T.V * 64);
  UP(static_cells, d->static_cells, (size_t)T.V * (T.S > 0 ? T.S : 1));
  UP(scan_order, d->scan_order, (size_t)T.V * T.D);
  UP(special_cells, d->special_cells, (size_t)T.V * 4 * CZ_MAX_SPECIAL);
  UP(static_masks, d->static_masks, (size_t)T.V * 8);
  UP(slot_type, d->slot_type, T.D);
  UP(type_flags, d->type_flags, T.T);
  UP(type_base, d->type_base, T.T);
  UP(type_count, d->type_count, T.T);
  UP(comp_slots, d->comp_slots, T.n_comp);
  UP(obs_table, d->obs_table, (size_t)T.V * 64 * T.tab_len);
  {  // float32 copies for cz_observe_f32 / CZ_STEP_OBS_F32: element-wise rounding of the f64 tables
    float xl[16], yl[16];
    for (int i = 0; i < 2 * T.W - 1; ++i) xl[i] = (float)d->xlut[i];
    for (int i = 0; i < 2 * T.H - 1; ++i) yl[i] = (float)d->ylut[i];
    UP(xlut32, xl, 2 * T.W - 1);
    UP(ylut32, yl, 2 * T.H - 1);
    const size_t n_tab = (size_t)T.V * 64 * T.tab_len;
    float* t32 = new (std::nothrow) float[n_tab ? n_tab : 1];
    if (!t32) { cz_tables_destroy(t); return cz_fail(CZ_EINVAL, "%s", "out of host memory"); }
    for (size_t i = 0; i < n_tab; ++i) t32[i] = (float)d->obs_table[i];
    UP(obs_table32, t32, n_tab);
    delete[] t32;
  }
  UP(recipe_nodes, d->recipe_nodes, (size_t)T.B * CZ_MAX_NODES);
  UP(recipe_len, d->recipe_len, T.B);
  uint32_t spans[256 * CZ_MAX_NODES];  // (stack: the library may be called from several host threads) per node: first slot | slots << 8 | required record bits << 16
  for (int b = 0; b < T.B; ++b)
    for (int k = 0; k < CZ_MAX_NODES; ++k) {
      const uint32_t node = d->recipe_nodes[b * CZ_MAX_NODES + k], ty = node & 255u, cond = (node >> 9) & 3u;
      uint32_t span = 0;
      if (!(node & 256u) && ty != 255u) {
        if ((int)ty >= T.T) {
          cz_tables_destroy(t);
          return cz_fail(CZ_EINVAL, "%s", "recipe node names a dynamic type outside type_base");
        }
        span = d->type_base[ty] | (uint32_t)d->type_count[ty] << 8;
      }
      spans[b * CZ_MAX_NODES + k] = span | (O_PRESENT | (cond == 1 ? O_CHOP : (cond == 2 ? O_MASH : 0u))) << 16;
    }
  UP(recipe_spans, spans, (size_t)T.B * CZ_MAX_NODES);
  UP(pool, d->pool, (size_t)T.P * T.rows);
  T.layout_cum = nullptr;
  if (d->layout_cum && rc == CZ_OK) {
    if (d->layout_cum[T.P - 1] != ~0ull) { cz_tables_destroy(t); return cz_fail(CZ_EINVAL, "%s", "layout_cum must end at 2^64 - 1"); }
    for (int i = 1; i < T.P; ++i)
      if (d->layout_cum[i] < d->layout_cum[i - 1]) { cz_tables_destroy(t); return cz_fail(CZ_EINVAL, "%s", "layout_cum must not decrease"); }
    UP(layout_cum, d->layout_cum, T.P);
    t->h_layout_cum = new (std::nothrow) uint64_t[T.P];
    if (!t->h_layout_cum) { cz_tables_destroy(t); return cz_fail(CZ_EINVAL, "%s", "out of host memory"); }
    memcpy(t->h_layout_cum, d->layout_cum, (size_t)T.P * sizeof(uint64_t));
  }
  UP(default_recipes, d->default_recipes, T.R);
  UP(spawn_x, d->spawn_x, (size_t)T.A * 8);
  UP(spawn_y, d->spawn_y, (size_t)T.A * 8);
  UP(spawn_n, d->spawn_n, (size_t)T.A * 2);
  if (rc == CZ_OK) {  // per-lane maps of the packed (observer, slot) layout
    int4 lm[64];  // entries 32-63: the second pair of a lane (kitchens with 33-64 (observer, slot) pairs)
    const int n0 = T.n_segs > 0 ? T.segs[0][1] >> 1 : 0, n1 = T.n_segs > 1 ? T.segs[1][1] >> 1 : 0;
    for (int l = 0; l < 64; ++l) {
      const bool live = T.n_comp > 0 && l < T.A * T.n_comp;
      int tt[2];
      for (int k = 0; k < 2; ++k) {
        const int e = (l & 31) + 32 * k;
        tt[k] = e < n0 ? (T.segs[0][0] >> 1) + e : (e < n0 + n1 ? (T.segs[1][0] >> 1) + e - n0 : -1);
      }
      // the computed-slot descriptor itself travels in the map: one load instead of a dependent pair
      lm[l] = make_int4(live ? (int)d->comp_slots[l % T.n_comp] : -1, live ? l / T.n_comp : 0, tt[0], tt[1]);
    }
    rc = upload(t, lm, 64, &T.lane_map);
  }
#undef UP
  if (rc == CZ_OK) {  // read-only shared-memory image of a block: LUTs + the small tables
    const size_t img_bytes = cz_block_smem_head(T.V);
    alignas(16) unsigned char img_buf[sizeof(BlockSmem) + CZ_SV * sizeof(VarTabs) + 16];
    memset(img_buf, 0, sizeof(img_buf));
    BlockSmem& img = *reinterpret_cast<BlockSmem*>(img_buf);
    for (int i = 0; i < 2 * T.W - 1; ++i) img.xlut[i] = d->xlut[i];
    for (int i = 0; i < 2 * T.H - 1; ++i) img.ylut[i] = d->ylut[i];
    SmemTabs& w = img.tabs;
    const int nv = T.V <= CZ_SV ? T.V : 1, nb = T.B < CZ_SB ? T.B : CZ_SB;
    for (int v = 0; v < nv; ++v) {
      VarTabs& x = w.var[v];
      for (int k = 0; k < 8; ++k) x.static_masks[k] = d->static_masks[v * 8 + k];
      for (int c = 0; c < 64; ++c) x.grid[c] = d->grid[v * 64 + c];
      for (int k = 0; k < T.D; ++k) x.scan_order[k] = d->scan_order[v * T.D + k];
      for (int k = 0; k < 4 * CZ_MAX_SPECIAL; ++k) x.special_cells[k] = d->special_cells[v * 4 * CZ_MAX_SPECIAL + k];
      for (int k = 0; k < T.S; ++k) x.static_cells[k] = d->static_cells[v * T.S + k];
    }
    for (int b = 0; b < nb; ++b) {
      for (int k = 0; k < CZ_MAX_NODES; ++k) {
        w.recipe_nodes[b][k] = d->recipe_nodes[b * CZ_MAX_NODES + k];
        w.recipe_spans[b][k] = spans[b * CZ_MAX_NODES + k];
      }
      w.recipe_len[b] = d->recipe_len[b];
      // descendants of every node (children come later in node_list, so one backward pass closes the relation)
      for (int k = CZ_MAX_NODES - 1; k >= 0; --k) {
        uint32_t desc = 1u << k;
        const uint32_t kids = d->recipe_nodes[b * CZ_MAX_NODES + k] >> 16;
        for (int j = k + 1; j < CZ_MAX_NODES; ++j)
          if (kids >> j & 1u) desc |= w.recipe_desc[b][j];
        w.recipe_desc[b][k] = (uint8_t)desc;
      }
    }
    for (int i = 0; i < T.D; ++i) { w.slot_type[i] = d->slot_type[i]; w.slot_tf[i] = d->type_flags[d->slot_type[i]]; }
    for (int i = 0; i < T.T; ++i) { w.type_base[i] = d->type_base[i]; w.type_count[i] = d->type_count[i]; }
    const unsigned char* dimg = nullptr;
    rc = upload(t, img_buf, img_bytes, &dimg);
    T.blob = dimg;
  }
  if (rc == CZ_OK) {  // grid observation: channel numbers of every dynamic slot (channel order in cz_b200.h)
    CzGridDev& g = t->grid;
    int n_chop = 0, n_mash = 0;
    for (int i = 0; i < T.T; ++i) {
      n_chop += (d->type_flags[i] & 2) != 0;
      n_mash += (d->type_flags[i] & 4) != 0;
    }
    uint32_t type_ch[CZ_MAX_TYPES], slot_ch[CZ_MAX_DYN];
    for (int i = 0, kc = 0, km = 0; i < T.T; ++i) {
      const uint32_t chop = (d->type_flags[i] & 2) ? (uint32_t)(12 + T.T + kc++) : 0u;
      const uint32_t mash = (d->type_flags[i] & 4) ? (uint32_t)(12 + T.T + n_chop + km++) : 0u;
      type_ch[i] = (uint32_t)(12 + i) | chop << 8 | mash << 16;
    }
    for (int s = 0; s < T.D; ++s) slot_ch[s] = d->slot_type[s] < T.T ? type_ch[d->slot_type[s]] : 0u;
    g.W = T.W; g.H = T.H; g.HW = T.W * T.H; g.D = T.D; g.rows = T.rows;
    g.G0 = 12 + T.T + n_chop + n_mash + 1;
    g.C = g.G0 + 7 * T.A;
    g.E = (uint32_t)(T.A * g.C * g.HW);
    g.grid = T.grid;
    rc = upload(t, slot_ch, T.D, &g.slot_ch);
  }
  if (rc != CZ_OK) { cz_tables_destroy(t); return rc; }
  size_t smem = cz_smem_bytes(T);
  if (smem > (size_t)prop.sharedMemPerBlockOptin) { cz_tables_destroy(t); return cz_fail(CZ_ELIMIT, "%s", "obs_len too large for shared memory staging"); }
  // the specialised kernels: one lane per (observer, slot) pair, one computed range, two table loads per
  // lane, small tables resident in shared memory
  const bool packed = T.n_comp > 0 && T.n_ranges == 1 && T.tab_len <= 128 && (T.L & 1) == 0 && T.V <= CZ_SV && T.B <= CZ_SB;
  t->simple = packed && T.A * T.n_comp <= 32;
  // 33-64 pairs (3-4 agent kitchens): specialised dynamics kernel + the warp-per-environment writer with two pairs per lane
  t->simple2 = packed && !t->simple && T.A * T.n_comp <= 64;
  {
    t->fast_dyn = T.V <= CZ_SV && T.B <= CZ_SB;
    const char* g = getenv("CZ_GENERIC");  // 1: everything generic; 2: only the observation plan (dynamics stay specialised)
    if (g && (g[0] == '1' || g[0] == '2')) t->simple = t->simple2 = 0;
    if (g && g[0] == '1') t->fast_dyn = 0;
    const char* k = getenv("CZ_TWO_KERNEL_MIN_ENVS");
    t->two_kernel_min_envs = k ? atoi(k) : 20480;  // measured crossover between 16384 and 24576 with the whole-row writer
                                                    // (profiles/microbench/inplace_path_sweep.py; 49152 with the round-1 writer)
    const char* aw = getenv("CZ_ANY_WRITER");
    t->any_writer = aw ? atoi(aw) : 1;
    const char* pod = getenv("CZ_POLICY_ON_DYN");
    t->policy_on_dyn = pod ? atoi(pod) : 1;
    const char* wr = getenv("CZ_WHOLE_ROWS");
    t->whole_rows = wr ? atoi(wr) : 15;
    const char* sp1 = getenv("CZ_SINGLE_PAIR");
    t->single_pair = sp1 ? atoi(sp1) : 1;
    const char* o32 = getenv("CZ_OBS32_PAIR");
    t->obs32_pair = o32 ? atoi(o32) : 1;
    const char* hc = getenv("CZ_HOST_CHUNKS");
    t->host_chunks = hc ? atoi(hc) : 4;
    if (t->host_chunks > 8) t->host_chunks = 8;
    const char* sp = getenv("CZ_SPLIT");
    t->split = sp ? atoi(sp) : 1;  // measured: every split is slower than the two plain launches (profiles/r02_notes.md)
    if (t->split > 8) t->split = 8;
    const char* wk = getenv("CZ_WARP_K_MAX_ENVS");
    t->warp_k_max_envs = wk ? atoi(wk) : 32768;
    const char* wg = getenv("CZ_WARP_GROUP");  // 16 or 32 lanes per environment in the warp kernel (default: 16 when D <= 16)
    t->warp_group = T.D <= 16 ? 16 : 32;
    if (wg && atoi(wg) == 32) t->warp_group = 32;
    // a single step goes to the warp kernel while the batch fits ONE wave of it (4 blocks x 8 environments per SM with
    // 16-lane groups, 7 x 4 with 32-lane groups: 4736 / 4144 environments on 148 SMs); the second wave doubles its time and
    // the fused lane-per-environment kernel wins (inplace_path_sweep.py: 4096 envs 10.8 vs 13.1 us, 6144 envs 18.3 vs 15.6 us)
    const char* w = getenv("CZ_WARP_MAX_ENVS");
    t->warp_max_envs = w ? atoi(w) : t->num_sms * (t->warp_group == 16 ? 32 : 28);
  }
#define SET_SMEM(K) CZ_CUDA(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prop.sharedMemPerBlockOptin))
#define SET_MODE(M)                                                                                    \
  SET_SMEM((cz_env_kernel<M, OBS_TMA, 0>)); SET_SMEM((cz_env_kernel<M, OBS_STG, 0>));                   \
  SET_SMEM((cz_env_kernel<M, OBS_TMA, 1>)); SET_SMEM((cz_env_kernel<M, OBS_TMA, 2>));                   \
  SET_SMEM((cz_env_kernel<M, OBS_TMA, 3>)); SET_SMEM((cz_env_kernel<M, OBS_TMA, 4>));                   \
  SET_SMEM((cz_env_kernel<M, OBS_STG, 1>)); SET_SMEM((cz_env_kernel<M, OBS_STG, 2>));                   \
  SET_SMEM((cz_env_kernel<M, OBS_STG, 3>)); SET_SMEM((cz_env_kernel<M, OBS_STG, 4>));                   \
  SET_SMEM((cz_env_kernel<M, OBS_NONE, 0>));                                                           \
  SET_SMEM((cz_env_kernel<M, OBS_NONE, 1>)); SET_SMEM((cz_env_kernel<M, OBS_NONE, 2>));                 \
  SET_SMEM((cz_env_kernel<M, OBS_NONE, 3>)); SET_SMEM((cz_env_kernel<M, OBS_NONE, 4>))
  SET_MODE(MODE_STEP); SET_MODE(MODE_RESET); SET_MODE(MODE_OBSERVE);
  SET_SMEM(cz_obs32_kernel);
  SET_SMEM(cz_obs_any_kernel<true>); SET_SMEM(cz_obs_any_kernel<false>); SET_SMEM(cz_obs_any_whole_kernel);
  SET_SMEM((cz_obs_whole_kernel<2, false>)); SET_SMEM((cz_obs_whole_kernel<3, false>)); SET_SMEM((cz_obs_whole_kernel<4, false>));
  SET_SMEM((cz_obs_whole_kernel<2, true>)); SET_SMEM((cz_obs_whole_kernel<3, true>)); SET_SMEM((cz_obs_whole_kernel<4, true>));
#define SET_WARP(S)                                                                                                     \
  SET_SMEM((cz_warp_kernel<1, 16, S>)); SET_SMEM((cz_warp_kernel<2, 16, S>)); SET_SMEM((cz_warp_kernel<3, 16, S>));    \
  SET_SMEM((cz_warp_kernel<4, 16, S>)); SET_SMEM((cz_warp_kernel<1, 32, S>)); SET_SMEM((cz_warp_kernel<2, 32, S>));    \
  SET_SMEM((cz_warp_kernel<3, 32, S>)); SET_SMEM((cz_warp_kernel<4, 32, S>))
  SET_WARP(false); SET_WARP(true);
#undef SET_WARP
#undef SET_MODE
#undef SET_SMEM
  *out = t;
  return CZ_OK;
}

extern "C" int cz_tables_destroy(cz_tables* t) {
  if (!t) return CZ_OK;
  cudaSetDevice(t->device);
  for (int i = 0; i < t->n_allocs; ++i) cudaFree(t->allocs[i]);
  if (t->d_actions) cudaFree(t->d_actions);
  if (t->d_obs) cudaFree(t->d_obs);
  if (t->d_reward) cudaFree(t->d_reward);
  if (t->d_term) cudaFree(t->d_term);
  if (t->d_trunc) cudaFree(t->d_trunc);
  if (t->d_rand) cudaFree(t->d_rand);
  if (t->d_keep) cudaFree(t->d_keep);
  delete[] t->h_layout_cum;
  if (t->pipe_ready) {
    cudaStreamDestroy(t->pipe_dyn); cudaStreamDestroy(t->pipe_obs);
    cudaEventDestroy(t->ev_user); cudaEventDestroy(t->ev_dyn);
    cudaEventDestroy(t->ev_pol_in); cudaEventDestroy(t->ev_pol_out);
    for (int c = 0; c < 4; ++c) cudaEventDestroy(t->ev_obs[c]);
    for (int c = 0; c < 8; ++c) cudaEventDestroy(t->ev_chunk[c]);
  }
  delete t;
  return CZ_OK;
}

extern "C" int cz_state_rows(const cz_tables* t) { return t ? t->dev.rows : CZ_EINVAL; }

// Environments per warp (log2): 32 for large batches; halved while the batch leaves SM schedulers without a warp
// (a step's latency is one warp's dynamics plus its observation loop, and the loop scales with the tile).
static int cz_tile_shift(const cz_tables* t, int n_envs) {
  int ts = 5;
  while (ts > 0 && ((n_envs + (1 << (ts - 1)) - 1) >> (ts - 1)) <= t->num_sms * 8) --ts;
  const char* f = getenv("CZ_TILE_SHIFT");
  if (f && f[0] >= '0' && f[0] <= '5') ts = f[0] - '0';
  return ts;
}

static int cz_grid(const cz_tables* t, int n_envs, int ts) {
  int tiles = (n_envs + (1 << ts) - 1) >> ts;
  int blocks = (tiles + CZ_WARPS_PER_BLOCK - 1) / CZ_WARPS_PER_BLOCK;
  // persistent tile loop beyond the blocks that are RESIDENT at once (CZ_MIN_BLOCKS per SM: 72 registers x 128 threads): with a
  // larger grid the surplus blocks start when the first ones have walked all their tiles and run alone on an idle GPU
  // (148 x 8 blocks for 1048576 environments: 0.87 of roofline in place against 0.93 with 148 x 7)
  int cap = t->num_sms * CZ_MIN_BLOCKS;
  return blocks < cap ? blocks : cap;
}

template <int MODE>
static int cz_launch(const cz_tables* t, const uint32_t* state, uint32_t* state_out, bool dyn_only, const uint8_t* actions,
                     const int32_t* layout_ids,
                     const uint8_t* recipe_ids, const uint8_t* mask, double* obs, double* reward, uint8_t* term,
                     uint8_t* trunc, uint32_t* err, int n_envs, uint32_t flags, uint64_t seed, int64_t env_offset,
                     void* stream, int ld = 0, int blocks_per_sm = 0) {
  if (ld <= 0) ld = n_envs;
  if (!t || !state || !state_out) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (MODE == MODE_OBSERVE && !obs) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (n_envs <= 0) return CZ_OK;
  if (!obs) dyn_only = true;  // no observation buffer: dynamics / reset only
  if (((uintptr_t)obs & 15) != 0) return cz_fail(CZ_EINVAL, "%s", "obs must be 16-byte aligned");
  size_t smem = cz_smem_bytes(t->dev);
  const int ts = cz_tile_shift(t, n_envs);
  int grid = cz_grid(t, n_envs, ts);
  // background dynamics of the pipelined step: a grid of `blocks_per_sm` blocks per SM walks the tiles in its
  // persistent loop, so the kernel keeps a few warp slots for a long time instead of half of every SM for a short one
  if (blocks_per_sm > 0 && grid > t->num_sms * blocks_per_sm) grid = t->num_sms * blocks_per_sm;
  flags = (flags & ~(7u << CZ_FLAG_TILE_SHIFT)) | ((uint32_t)ts << CZ_FLAG_TILE_SHIFT);
  cudaStream_t s = (cudaStream_t)stream;
#define CZ_GO(O, NA)                                                                                                  \
  cz_env_kernel<MODE, O, NA><<<grid, CZ_THREADS, smem, s>>>(t->dev, state, state_out, actions, layout_ids, recipe_ids, mask, obs, \
                                                           reward, term, trunc, err, n_envs, flags, seed, env_offset, ld)
  if (dyn_only && (t->simple || t->simple2 || t->fast_dyn)) {
    switch (t->dev.A) {
      case 1: CZ_GO(OBS_NONE, 1); break;
      case 2: CZ_GO(OBS_NONE, 2); break;
      case 3: CZ_GO(OBS_NONE, 3); break;
      default: CZ_GO(OBS_NONE, 4); break;
    }
  } else if (dyn_only) {
    CZ_GO(OBS_NONE, 0);
  } else if (t->simple && t->obs_path == OBS_TMA) {
    switch (t->dev.A) {
      case 1: CZ_GO(OBS_TMA, 1); break;
      case 2: CZ_GO(OBS_TMA, 2); break;
      case 3: CZ_GO(OBS_TMA, 3); break;
      default: CZ_GO(OBS_TMA, 4); break;
    }
  } else if (t->simple) {
    switch (t->dev.A) {
      case 1: CZ_GO(OBS_STG, 1); break;
      case 2: CZ_GO(OBS_STG, 2); break;
      case 3: CZ_GO(OBS_STG, 3); break;
      default: CZ_GO(OBS_STG, 4); break;
    }
  } else if (t->obs_path == OBS_TMA) {
    CZ_GO(OBS_TMA, 0);
  } else {
    CZ_GO(OBS_STG, 0);
  }
#undef CZ_GO
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}

// The warp-per-environment float64 row writer (packed plans) on `s`.
// `alone`: nothing else is meant to share the SMs with this launch (in-place step, cz_observe) — see cz_launch_obs32
static int cz_launch_obs64(const cz_tables* t, const uint32_t* state, double* obs, int n_envs, cudaStream_t s, int ld = 0,
                           bool alone = false) {
  if (ld <= 0) ld = n_envs;
  if (!state || !obs) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (((uintptr_t)obs & 15) != 0) return cz_fail(CZ_EINVAL, "%s", "obs must be 16-byte aligned");
  if (n_envs <= 0) return CZ_OK;
  if ((t->simple || (t->simple2 && (t->whole_rows & 4))) && t->dev.A >= 2 && (t->whole_rows & (alone ? 1 : 2)) &&
      n_envs >= ENVS_WARPS * t->num_sms) {
    const size_t smem = (size_t)ENVS_WARPS * t->dev.A * t->dev.L * 8;  // the A whole rows of one environment per warp
    if (smem <= t->smem_optin) {
      const int blocks = (n_envs + ENVS_WARPS - 1) / ENVS_WARPS;
#define CZ_WHOLE_GO(NA)                                                                                                   \
  if (t->simple2) cz_obs_whole_kernel<NA, true><<<blocks, 32 * ENVS_WARPS, smem, s>>>(t->dev, state, obs, n_envs, ld);    \
  else cz_obs_whole_kernel<NA, false><<<blocks, 32 * ENVS_WARPS, smem, s>>>(t->dev, state, obs, n_envs, ld)
      switch (t->dev.A) {
        case 2: CZ_WHOLE_GO(2); break;
        case 3: CZ_WHOLE_GO(3); break;
        default: CZ_WHOLE_GO(4); break;
      }
#undef CZ_WHOLE_GO
      g_launches.fetch_add(1);
      CZ_CUDA(cudaGetLastError());
      return CZ_OK;
    }
  }
  if (alone && t->simple && t->dev.A == 1 && t->single_pair && n_envs >= 2 * ENVS_WARPS * t->num_sms) {
    const size_t smem = (size_t)ENVS_WARPS * 2 * t->dev.L * 8;  // two whole rows per warp
    if (smem <= 48 * 1024) {
      const int blocks = (n_envs + 2 * ENVS_WARPS - 1) / (2 * ENVS_WARPS);
      cz_obs_single_pair_kernel<<<blocks, 32 * ENVS_WARPS, smem, s>>>(t->dev, state, obs, n_envs, ld);
      g_launches.fetch_add(1);
      CZ_CUDA(cudaGetLastError());
      return CZ_OK;
    }
  }
  const int blocks = (n_envs + ENVS_WARPS - 1) / ENVS_WARPS;
  const size_t smem = (size_t)ENVS_WARPS * t->dev.A * ((t->dev.stage_len + 1) / 2) * 16;
#define CZ_OBS_GO(NA)                                                                                               \
  if (t->simple2) cz_obs_envs_kernel<NA, true><<<blocks, 32 * ENVS_WARPS, smem, s>>>(t->dev, state, obs, n_envs, ld); \
  else cz_obs_envs_kernel<NA, false><<<blocks, 32 * ENVS_WARPS, smem, s>>>(t->dev, state, obs, n_envs, ld)
  switch (t->dev.A) {
    case 1: CZ_OBS_GO(1); break;
    case 2: CZ_OBS_GO(2); break;
    case 3: CZ_OBS_GO(3); break;
    default: CZ_OBS_GO(4); break;
  }
#undef CZ_OBS_GO
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}

// The any-plan float64 row writer (tables outside the packed class) on `s`.
static int cz_launch_obs_any(const cz_tables* t, const uint32_t* state, double* obs, int n_envs, cudaStream_t s, int ld = 0) {
  if (!state || !obs) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (n_envs <= 0) return CZ_OK;
  if (ld <= 0) ld = n_envs;
  const CzDev& T = t->dev;
  if ((t->whole_rows & 8) && ((T.A * T.L) & 1) == 0 && ((uintptr_t)obs & 15) == 0) {  // whole rows staged, one bulk store per environment
    const size_t pw = (size_t)T.A * T.L * sizeof(double);
    int warps = (int)(((size_t)72 * 1024) / pw);  // at least three blocks per SM stay resident
    if (warps > ENVS_WARPS) warps = ENVS_WARPS;
    if (warps >= 1) {
      const int blocks = (n_envs + warps - 1) / warps;
      cz_obs_any_whole_kernel<<<blocks, 32 * ENVS_WARPS, pw * warps, s>>>(t->dev, state, obs, n_envs, ld, warps);
      g_launches.fetch_add(1);
      CZ_CUDA(cudaGetLastError());
      return CZ_OK;
    }
  }
  const size_t per_warp = (size_t)T.A * ((T.stage_len + 1) & ~1) * sizeof(double);
  int warps = per_warp ? (int)(((size_t)96 * 1024) / per_warp) : ENVS_WARPS;  // at least two blocks per SM stay resident
  if (warps > ENVS_WARPS) warps = ENVS_WARPS;
  if (warps < 1) warps = 1;
  const size_t smem = per_warp * warps;
  if (smem > t->smem_optin) return cz_fail(CZ_ELIMIT, "%s", "observation rows too long for the row writer");
  const int blocks = (n_envs + warps - 1) / warps;
  if ((T.L & 1) == 0) cz_obs_any_kernel<true><<<blocks, 32 * ENVS_WARPS, smem, s>>>(t->dev, state, obs, n_envs, ld, warps);
  else cz_obs_any_kernel<false><<<blocks, 32 * ENVS_WARPS, smem, s>>>(t->dev, state, obs, n_envs, ld, warps);
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}

extern "C" int cz_reset(const cz_tables* t, uint32_t* state, const int32_t* layout_ids, const uint8_t* recipe_ids,
                        const uint8_t* mask, double* obs, uint32_t* error_flags, int n_envs, void* stream) {
  if (!layout_ids) return cz_fail(CZ_EINVAL, "%s", "layout_ids is required");
  if (t && t->simple2 && obs && !mask) {  // state first, then every row (a masked reset takes the generic kernel below)
    int rc = cz_launch<MODE_RESET>(t, state, state, true, nullptr, layout_ids, recipe_ids, mask, nullptr, nullptr, nullptr, nullptr,
                                   error_flags, n_envs, 0, 0, 0, stream);
    if (rc != CZ_OK) return rc;
    return cz_launch_obs64(t, state, obs, n_envs, (cudaStream_t)stream);
  }
  return cz_launch<MODE_RESET>(t, state, state, false, nullptr, layout_ids, recipe_ids, mask, obs, nullptr, nullptr, nullptr, error_flags,
                               n_envs, 0, 0, 0, stream);
}

// default layout ids of an episode: cz_layout_draw(seed, env_offset + e, episode) % P for every environment
__global__ void cz_layout_ids_kernel(int32_t* __restrict__ out, int n_envs, const uint64_t* __restrict__ cum, int P, uint64_t seed,
                                     int64_t env_offset, uint64_t episode) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n_envs) out[e] = (int32_t)cz_pick_layout(cum, P, cz_mix(seed, (uint64_t)(env_offset + e), episode));
}

extern "C" int cz_layout_ids(const cz_tables* t, int32_t* layout_ids, int n_envs, uint64_t seed, int64_t env_offset, uint64_t episode,
                             void* stream) {
  if (!t || !layout_ids) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (n_envs <= 0) return CZ_OK;
  cz_layout_ids_kernel<<<(n_envs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(layout_ids, n_envs, t->dev.layout_cum, t->dev.P, seed, env_offset,
                                                                               episode);
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}

extern "C" int cz_random_actions(const cz_tables* t, uint8_t* actions, int n_envs, uint64_t seed, uint64_t step,
                                 int64_t env_offset, void* stream);

static int cz_pipe_init(cz_tables* t);

// ---- episode statistics (cz_stats.cuh) ------------------------------------------------------------------------------
extern "C" int cz_stats_attach(cz_tables* t, const cz_stats_desc* d) {
  if (!t) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (!d) {
    memset(&t->stats, 0, sizeof(t->stats));
    return CZ_OK;
  }
  if (d->n_envs < 1 || !d->ret || !d->episode || !d->open || !d->last_ret || !d->last_len || !d->last_served ||
      !d->last_success || !d->finished || !d->totals)
    return cz_fail(CZ_EINVAL, "%s", "cz_stats_attach: every buffer is required and n_envs must be at least 1");
  CzStatsDev& S = t->stats;
  S.ret = d->ret; S.episode = d->episode; S.open = d->open; S.last_ret = d->last_ret; S.last_len = d->last_len;
  S.last_served = d->last_served; S.last_success = d->last_success; S.finished = d->finished; S.totals = d->totals;
  S.n = d->n_envs;
  return CZ_OK;
}

// CZ_STEP_EPISODE_STATS needs attached statistics of exactly this batch
static int cz_stats_check(const cz_tables* t, int n_envs) {
  if (t->stats.n == 0) return cz_fail(CZ_EINVAL, "%s", "CZ_STEP_EPISODE_STATS without statistics attached (cz_stats_attach)");
  if (t->stats.n != n_envs) return cz_fail(CZ_EINVAL, "%s", "CZ_STEP_EPISODE_STATS: n_envs differs from the attached statistics");
  return CZ_OK;
}

// the record update after one step of all n_envs environments of `state` (post-step state, reward of that step)
static int cz_stats_launch(const cz_tables* t, const uint32_t* state, const double* reward, int n_envs, cudaStream_t s) {
  const CzDev& T = t->dev;
  const uint32_t* misc = state + (size_t)(T.D + T.A) * n_envs;
  const int blocks = (n_envs + CZ_STATS_THREADS - 1) / CZ_STATS_THREADS;
  switch (T.A) {
    case 1: cz_stats_kernel<1><<<blocks, CZ_STATS_THREADS, 0, s>>>(t->stats, misc, reward, n_envs, n_envs, T.R, T.end_all); break;
    case 2: cz_stats_kernel<2><<<blocks, CZ_STATS_THREADS, 0, s>>>(t->stats, misc, reward, n_envs, n_envs, T.R, T.end_all); break;
    case 3: cz_stats_kernel<3><<<blocks, CZ_STATS_THREADS, 0, s>>>(t->stats, misc, reward, n_envs, n_envs, T.R, T.end_all); break;
    default: cz_stats_kernel<4><<<blocks, CZ_STATS_THREADS, 0, s>>>(t->stats, misc, reward, n_envs, n_envs, T.R, T.end_all); break;
  }
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}

extern "C" int cz_stats_clear(const cz_tables* t, const uint32_t* state, int n_envs, void* stream) {
  if (!t || !state) return cz_fail(CZ_EINVAL, "%s", "null argument");
  int rc = cz_stats_check(t, n_envs);
  if (rc != CZ_OK) return rc;
  const CzDev& T = t->dev;
  const int blocks = (n_envs + CZ_STATS_THREADS - 1) / CZ_STATS_THREADS;
  cz_stats_clear_kernel<<<blocks, CZ_STATS_THREADS, 0, (cudaStream_t)stream>>>(t->stats, state + (size_t)(T.D + T.A) * n_envs,
                                                                               n_envs, n_envs, T.A);
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}

// In-place step of a large batch as `split` column ranges: the dynamics of range c + 1 (internal high-priority stream)
// run under the row writer of range c (second internal stream), so only the first range's dynamics are exposed.  The
// caller's stream forks into both and joins them again: every output is ordered on it when the call's work is done,
// exactly like the two launches it replaces.
static int cz_step_split(cz_tables* t, uint32_t* state, const uint8_t* actions, double* obs, double* reward,
                         uint8_t* terminated, uint8_t* truncated, uint32_t* error_flags, int n_envs, uint32_t flags,
                         uint64_t seed, int64_t env_offset, void* stream, bool stats) {
  int rc = cz_pipe_init(t);
  if (rc != CZ_OK) return rc;
  const int A = t->dev.A, L = t->dev.L;
  const int chunk = (((n_envs + t->split - 1) / t->split) + 255) & ~255;  // whole tiles and whole writer blocks
  cudaStream_t user = (cudaStream_t)stream;
  CZ_CUDA(cudaEventRecord(t->ev_user, user));
  CZ_CUDA(cudaStreamWaitEvent(t->pipe_dyn, t->ev_user, 0));
  CZ_CUDA(cudaStreamWaitEvent(t->pipe_obs, t->ev_user, 0));
  int c = 0;
  for (int e0 = 0; e0 < n_envs; e0 += chunk, ++c) {
    const int n = n_envs - e0 < chunk ? n_envs - e0 : chunk;
    const size_t na = (size_t)e0 * A;
    rc = cz_launch<MODE_STEP>(t, state + e0, state + e0, true, actions + na, nullptr, nullptr, nullptr, nullptr, reward + na,
                              terminated + na, truncated + na, error_flags ? error_flags + e0 : nullptr, n, flags, seed,
                              env_offset + e0, t->pipe_dyn, n_envs);
    if (rc != CZ_OK) return rc;
    CZ_CUDA(cudaEventRecord(t->ev_chunk[c], t->pipe_dyn));
    CZ_CUDA(cudaStreamWaitEvent(t->pipe_obs, t->ev_chunk[c], 0));
    rc = cz_launch_obs64(t, state + e0, obs + na * L, n, t->pipe_obs, n_envs);
    if (rc != CZ_OK) return rc;
  }
  if (stats) {  // one launch over all n after every range's dynamics, before the event the caller's stream waits on
    rc = cz_stats_launch(t, state, reward, n_envs, t->pipe_dyn);
    if (rc != CZ_OK) return rc;
  }
  CZ_CUDA(cudaEventRecord(t->ev_dyn, t->pipe_dyn));
  CZ_CUDA(cudaEventRecord(t->ev_obs[0], t->pipe_obs));
  CZ_CUDA(cudaStreamWaitEvent(user, t->ev_dyn, 0));
  CZ_CUDA(cudaStreamWaitEvent(user, t->ev_obs[0], 0));
  return CZ_OK;
}

// one in-place step with resident actions on the lane-per-environment kernels
static int cz_step_kernels(const cz_tables* t, uint32_t* state, const uint8_t* actions, double* obs, double* reward,
                           uint8_t* terminated, uint8_t* truncated, uint32_t* error_flags, int n_envs, uint32_t flags,
                           uint64_t seed, int64_t env_offset, void* stream, bool stats, bool* stats_done) {
  // 33-64 pair plans always, and large batches of the other packed plans (the short-block row writer streams faster than the
  // observation phase of the fused kernel; small batches keep the single launch): dynamics, then the row writer
  if (t && obs && !(flags & CZ_STEP_OBS_F32) &&
      (t->simple2 || (t->simple && t->two_kernel_min_envs > 0 && n_envs >= t->two_kernel_min_envs))) {
    if (t->split > 1 && n_envs >= 2 * t->two_kernel_min_envs && t->two_kernel_min_envs > 0) {
      *stats_done = stats;  // the split step updates the statistics on its dynamics stream
      return cz_step_split(const_cast<cz_tables*>(t), state, actions, obs, reward, terminated, truncated, error_flags, n_envs, flags,
                           seed, env_offset, stream, stats);
    }
    int rc = cz_launch<MODE_STEP>(t, state, state, true, actions, nullptr, nullptr, nullptr, nullptr, reward, terminated, truncated,
                                  error_flags, n_envs, flags, seed, env_offset, stream);
    if (rc != CZ_OK) return rc;
    return cz_launch_obs64(t, state, obs, n_envs, (cudaStream_t)stream, 0, true);
  }
  // tables outside the packed class, large batches: the generic dynamics kernel, then the any-plan row writer (short
  // blocks stream faster than the fused kernel's observation phase, as for the packed plans)
  if (t && obs && !(flags & CZ_STEP_OBS_F32) && !t->simple && !t->simple2 && t->two_kernel_min_envs > 0 &&
      n_envs >= t->two_kernel_min_envs && t->any_writer) {
    int rc = cz_launch<MODE_STEP>(t, state, state, true, actions, nullptr, nullptr, nullptr, nullptr, reward, terminated, truncated,
                                  error_flags, n_envs, flags, seed, env_offset, stream);
    if (rc != CZ_OK) return rc;
    return cz_launch_obs_any(t, state, obs, n_envs, (cudaStream_t)stream);
  }
  if ((flags & CZ_STEP_OBS_F32) && obs) {  // dynamics, then the float32 row writer on the same stream
    int rc = cz_launch<MODE_STEP>(t, state, state, true, actions, nullptr, nullptr, nullptr, nullptr, reward, terminated, truncated,
                                  error_flags, n_envs, flags, seed, env_offset, stream);
    if (rc != CZ_OK) return rc;
    return cz_launch_obs32(t, state, reinterpret_cast<float*>(obs), n_envs, (cudaStream_t)stream);
  }
  return cz_launch<MODE_STEP>(t, state, state, false, actions, nullptr, nullptr, nullptr, obs, reward, terminated, truncated,
                              error_flags, n_envs, flags, seed, env_offset, stream);
}

// one in-place step on the per-step kernels; with `stats`, the record update follows the step's kernels on `stream` (the
// split step launches it itself, on its dynamics stream)
static int cz_step_one(const cz_tables* t, uint32_t* state, const uint8_t* actions, double* obs, double* reward,
                       uint8_t* terminated, uint8_t* truncated, uint32_t* error_flags, int n_envs, uint32_t flags,
                       uint64_t seed, int64_t env_offset, void* stream, bool stats) {
  bool stats_done = false;
  int rc = cz_step_kernels(t, state, actions, obs, reward, terminated, truncated, error_flags, n_envs, flags, seed, env_offset,
                           stream, stats, &stats_done);
  if (rc != CZ_OK || !stats || stats_done) return rc;
  return cz_stats_launch(t, state, reward, n_envs, (cudaStream_t)stream);
}

// k_steps consecutive steps of every environment in ONE launch of the warp-per-environment kernel
static int cz_launch_warp(const cz_tables* t, uint32_t* state, const uint8_t* actions, double* obs, double* reward,
                          uint8_t* terminated, uint8_t* truncated, uint32_t* error_flags, int n_envs, int k_steps, uint32_t flags,
                          uint64_t seed, int64_t env_offset, uint64_t action_step, void* stream, bool stats) {
  if (((uintptr_t)obs & 15) != 0) return cz_fail(CZ_EINVAL, "%s", "obs must be 16-byte aligned");
  const CzDev& T = t->dev;
  // two environments per warp (16-lane groups) when every dynamic slot finds a lane in half a warp
  const int G = t->warp_group;
  const int groups = WK_WARPS * 32 / G;
  const int blocks = (n_envs + groups - 1) / groups;
  const size_t smem = wk_smem_bytes(T.V, T.A, CZ_WARP_WHOLE ? T.L : T.stage_len, G);
  cudaStream_t s = (cudaStream_t)stream;
#define CZ_WARP_GO_S(NA, S)                                                                                                    \
  if (G == 16)                                                                                                                 \
    cz_warp_kernel<NA, 16, S><<<blocks, 32 * WK_WARPS, smem, s>>>(t->dev, state, actions, obs, reward, terminated, truncated,   \
                                                                  error_flags, n_envs, k_steps, flags, seed, env_offset,         \
                                                                  action_step, t->stats);                                        \
  else                                                                                                                         \
    cz_warp_kernel<NA, 32, S><<<blocks, 32 * WK_WARPS, smem, s>>>(t->dev, state, actions, obs, reward, terminated, truncated,   \
                                                                  error_flags, n_envs, k_steps, flags, seed, env_offset,         \
                                                                  action_step, t->stats)
#define CZ_WARP_GO(NA)          \
  if (stats) {                  \
    CZ_WARP_GO_S(NA, true);     \
  } else {                      \
    CZ_WARP_GO_S(NA, false);    \
  }
  switch (T.A) {
    case 1: CZ_WARP_GO(1); break;
    case 2: CZ_WARP_GO(2); break;
    case 3: CZ_WARP_GO(3); break;
    default: CZ_WARP_GO(4); break;
  }
#undef CZ_WARP_GO
#undef CZ_WARP_GO_S
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}

extern "C" int cz_step(const cz_tables* t, uint32_t* state, const uint8_t* actions, double* obs, double* reward,
                       uint8_t* terminated, uint8_t* truncated, uint32_t* error_flags, int n_envs, int k_steps, uint32_t flags,
                       uint64_t seed, int64_t env_offset, uint64_t action_step, void* stream) {
  if (!t || !state || !reward || !terminated || !truncated) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (k_steps < 1) return cz_fail(CZ_EINVAL, "%s", "k_steps must be at least 1");
  const bool dev_actions = (flags & CZ_STEP_DEVICE_ACTIONS) != 0;
  if (!actions && !dev_actions) return cz_fail(CZ_EINVAL, "%s", "actions is NULL and CZ_STEP_DEVICE_ACTIONS is not set");
  if (dev_actions) actions = nullptr;
  const bool stats = (flags & CZ_STEP_EPISODE_STATS) != 0;
  if (stats) {
    int rc = cz_stats_check(t, n_envs);
    if (rc != CZ_OK) return rc;
    flags &= ~CZ_STEP_EPISODE_STATS;
  }
  if (n_envs <= 0) return CZ_OK;
  const CzDev& T = t->dev;
  const bool warp_ok = (t->simple || t->simple2) && !(flags & CZ_STEP_OBS_F32);
  if (warp_ok && (k_steps > 1 ? n_envs <= t->warp_k_max_envs : n_envs <= t->warp_max_envs))
    return cz_launch_warp(t, state, actions, obs, reward, terminated, truncated, error_flags, n_envs, k_steps, flags, seed,
                          env_offset, action_step, stream, stats);
  // everything else (generic tables, float32 rows, large batches): k_steps launches of the per-step kernels
  cz_tables* tm = const_cast<cz_tables*>(t);
  if (dev_actions && n_envs > t->rand_envs) {
    if (tm->d_rand) cudaFree(tm->d_rand);
    tm->rand_envs = 0;
    CZ_CUDA(cudaMalloc((void**)&tm->d_rand, (size_t)n_envs * T.A));
    tm->rand_envs = n_envs;
  }
  const size_t na = (size_t)n_envs * T.A;
  const bool keep = (flags & CZ_STEP_KEEP_ALL) != 0 && k_steps > 1;
  const size_t obs_bytes = na * T.L * ((flags & CZ_STEP_OBS_F32) ? sizeof(float) : sizeof(double));
  for (int k = 0; k < k_steps; ++k) {
    const uint8_t* a = actions ? actions + (size_t)k * na : t->d_rand;
    if (dev_actions) {
      int rc = cz_random_actions(t, tm->d_rand, n_envs, seed, action_step + (uint64_t)k, env_offset, stream);
      if (rc != CZ_OK) return rc;
    }
    const size_t o = keep ? (size_t)k : 0;
    double* obs_k = obs ? reinterpret_cast<double*>(reinterpret_cast<char*>(obs) + o * obs_bytes) : nullptr;
    // KEEP_ALL: step k's rows start k * obs_bytes into the buffer, which is 16-byte aligned only when obs_bytes is a multiple
    // of 16 (odd n * A * L in float64, n * A * L not a multiple of 4 in float32); the row writers need 16-byte aligned rows,
    // so such a step writes into aligned scratch that is then copied into place
    double* dst = obs_k;
    if (obs_k && ((uintptr_t)obs_k & 15) != 0) {
      if (obs_bytes > t->keep_bytes) {
        if (tm->d_keep) cudaFree(tm->d_keep);
        tm->d_keep = nullptr;
        tm->keep_bytes = 0;
        CZ_CUDA(cudaMalloc(&tm->d_keep, obs_bytes));
        tm->keep_bytes = obs_bytes;
      }
      obs_k = reinterpret_cast<double*>(tm->d_keep);
    }
    int rc = cz_step_one(t, state, a, obs_k, reward + o * na, terminated + o * na, truncated + o * na, error_flags, n_envs,
                         flags & ~(CZ_STEP_DEVICE_ACTIONS | CZ_STEP_KEEP_ALL), seed, env_offset, stream, stats);
    if (rc != CZ_OK) return rc;
    if (dst != obs_k) CZ_CUDA(cudaMemcpyAsync(dst, obs_k, obs_bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  }
  return CZ_OK;
}

extern "C" int cz_observe_f32(const cz_tables* t, const uint32_t* state, float* obs32, int n_envs, void* stream) {
  return cz_launch_obs32(t, state, obs32, n_envs, (cudaStream_t)stream);
}

extern "C" int cz_observe(const cz_tables* t, const uint32_t* state, double* obs, int n_envs, void* stream) {
  if (t && (t->simple2 || (t->simple && t->two_kernel_min_envs > 0 && n_envs >= t->two_kernel_min_envs)))
    return cz_launch_obs64(t, state, obs, n_envs, (cudaStream_t)stream, 0, true);  // the short-block row writer (as in cz_step)
  if (t && !t->simple && !t->simple2 && t->any_writer && t->two_kernel_min_envs > 0 && n_envs >= t->two_kernel_min_envs)
    return cz_launch_obs_any(t, state, obs, n_envs, (cudaStream_t)stream);
  return cz_launch<MODE_OBSERVE>(t, state, const_cast<uint32_t*>(state), false, nullptr, nullptr, nullptr, nullptr, obs, nullptr,
                                 nullptr, nullptr, nullptr, n_envs, 0, 0, 0, stream);
}

extern "C" int cz_grid_channels(const cz_tables* t) {
  if (!t) return cz_fail(CZ_EINVAL, "%s", "null argument");
  return t->grid.C;
}

extern "C" int cz_observe_grid(const cz_tables* t, const uint32_t* state, uint8_t* grid, int n_envs, void* stream) {
  if (!t || !state || !grid) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (n_envs <= 0) return CZ_OK;
  const CzGridDev& G = t->grid;
  int warps = (int)(GRID_SMEM_BUDGET / G.E);  // E <= 4 agents x 89 channels x 64 cells = 22784 bytes: at least one
  if (warps > GRID_WARPS) warps = GRID_WARPS;
  if (warps < 1) warps = 1;
  const size_t smem = ((size_t)warps * G.E + 30) & ~(size_t)15;  // up to 15 bytes of shift in front, rounded up to 16
  const int blocks = (n_envs + warps - 1) / warps;
  cudaStream_t s = (cudaStream_t)stream;
  switch (t->dev.A) {
    case 1: cz_grid_kernel<1><<<blocks, 32 * warps, smem, s>>>(G, state, grid, n_envs, warps); break;
    case 2: cz_grid_kernel<2><<<blocks, 32 * warps, smem, s>>>(G, state, grid, n_envs, warps); break;
    case 3: cz_grid_kernel<3><<<blocks, 32 * warps, smem, s>>>(G, state, grid, n_envs, warps); break;
    default: cz_grid_kernel<4><<<blocks, 32 * warps, smem, s>>>(G, state, grid, n_envs, warps); break;
  }
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}

static int cz_pipe_init(cz_tables* t) {
  if (t->pipe_ready) return CZ_OK;
  int lo = 0, hi = 0;
  CZ_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  const char* sw = getenv("CZ_PIPE_PRIO");  // "swap": row writer above the dynamics, "equal": same priority (A/B only)
  const int p_dyn = (sw && !strcmp(sw, "swap")) ? lo : hi, p_obs = (sw && !strcmp(sw, "swap")) ? hi : ((sw && !strcmp(sw, "equal")) ? hi : lo);
  CZ_CUDA(cudaStreamCreateWithPriority(&t->pipe_dyn, cudaStreamNonBlocking, p_dyn));  // highest priority: slips in between observe blocks
  CZ_CUDA(cudaStreamCreateWithPriority(&t->pipe_obs, cudaStreamNonBlocking, p_obs));
  CZ_CUDA(cudaEventCreateWithFlags(&t->ev_user, cudaEventDisableTiming));
  CZ_CUDA(cudaEventCreateWithFlags(&t->ev_dyn, cudaEventDisableTiming));
  for (int c = 0; c < 4; ++c) CZ_CUDA(cudaEventCreateWithFlags(&t->ev_obs[c], cudaEventDisableTiming));
  for (int c = 0; c < 8; ++c) CZ_CUDA(cudaEventCreateWithFlags(&t->ev_chunk[c], cudaEventDisableTiming));
  CZ_CUDA(cudaEventCreateWithFlags(&t->ev_pol_in, cudaEventDisableTiming));
  CZ_CUDA(cudaEventCreateWithFlags(&t->ev_pol_out, cudaEventDisableTiming));
  t->pipe_ready = 1;
  return CZ_OK;
}

extern "C" int cz_pipeline_config(cz_tables* t, int n_buffers, int dyn_blocks_per_sm) {
  if (!t || n_buffers < 2 || n_buffers > 4 || dyn_blocks_per_sm < 0 || dyn_blocks_per_sm > 8)
    return cz_fail(CZ_EINVAL, "%s", "cz_pipeline_config: 2..4 buffers, 0..8 dynamics blocks per SM");
  int rc = cz_pipeline_reset(t, 0);  // drains the internal streams
  if (rc != CZ_OK) return rc;
  t->pipe_buffers = n_buffers;
  t->pipe_dyn_blocks = dyn_blocks_per_sm;
  return CZ_OK;
}

extern "C" int cz_pipeline_reset(cz_tables* t, int current_half) {
  if (!t || current_half < 0 || current_half >= (t->pipe_buffers ? t->pipe_buffers : 2)) return cz_fail(CZ_EINVAL, "%s", "bad argument");
  int rc = cz_pipe_init(t);
  if (rc != CZ_OK) return rc;
  CZ_CUDA(cudaStreamSynchronize(t->pipe_dyn));
  CZ_CUDA(cudaStreamSynchronize(t->pipe_obs));
  t->pipe_cur = current_half;
  for (int c = 0; c < 4; ++c) t->pipe_obs_pending[c] = 0;
  t->pipe_steps = 0;
  return CZ_OK;
}

extern "C" int cz_pipeline_current(const cz_tables* t) { return t ? t->pipe_cur : CZ_EINVAL; }

extern "C" int cz_step_pipelined(cz_tables* t, uint32_t* state2, const uint8_t* actions, double* obs, double* reward,
                                 uint8_t* terminated, uint8_t* truncated, uint32_t* error_flags, int n_envs, uint32_t flags,
                                 uint64_t seed, int64_t env_offset, void* stream) {
  if (!t || !state2 || !actions || !obs || !reward || !terminated || !truncated) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (!t->simple && !t->simple2) return cz_fail(CZ_EINVAL, "%s", "the pipelined step needs the specialised kernels (see DESIGN.md)");
  const bool stats = (flags & CZ_STEP_EPISODE_STATS) != 0;
  if (stats) {
    int rc = cz_stats_check(t, n_envs);
    if (rc != CZ_OK) return rc;
    flags &= ~CZ_STEP_EPISODE_STATS;
  }
  int rc = cz_pipe_init(t);
  if (rc != CZ_OK) return rc;
  const size_t half = (size_t)t->dev.rows * n_envs;
  const int cur = t->pipe_cur, nxt = (cur + 1) % t->pipe_buffers;
  uint32_t* in = state2 + (size_t)cur * half;
  uint32_t* out = state2 + (size_t)nxt * half;
  cudaStream_t user = (cudaStream_t)stream;
  // the caller's stream has produced the actions and consumed the previous rewards / flags
  CZ_CUDA(cudaEventRecord(t->ev_user, user));
  CZ_CUDA(cudaStreamWaitEvent(t->pipe_dyn, t->ev_user, 0));
  // the observe kernel that read the half we are about to overwrite must be done
  if (t->pipe_obs_pending[nxt]) CZ_CUDA(cudaStreamWaitEvent(t->pipe_dyn, t->ev_obs[nxt], 0));
  rc = cz_launch<MODE_STEP>(t, in, out, true, actions, nullptr, nullptr, nullptr, obs, reward, terminated, truncated,
                            error_flags, n_envs, flags, seed, env_offset, t->pipe_dyn, 0,
                            t->pipe_steps == 0 ? 0 : t->pipe_dyn_blocks);  // nothing to hide behind on the first step: full grid
  if (rc != CZ_OK) return rc;
  if (stats) {  // on the dynamics stream, before the event that orders the caller's stream: ordered like rewards and flags
    rc = cz_stats_launch(t, out, reward, n_envs, t->pipe_dyn);
    if (rc != CZ_OK) return rc;
  }
  CZ_CUDA(cudaEventRecord(t->ev_dyn, t->pipe_dyn));
  CZ_CUDA(cudaStreamWaitEvent(t->pipe_obs, t->ev_dyn, 0));
  CZ_CUDA(cudaStreamWaitEvent(t->pipe_obs, t->ev_user, 0));
  // the caller's stream trails the dynamics: whatever it does next (overwrite or free the action buffer, read the
  // rewards / flags / state, run a policy) is ordered after this step's dynamics; only the rows need cz_pipeline_wait
  CZ_CUDA(cudaStreamWaitEvent(user, t->ev_dyn, 0));
  if (flags & CZ_STEP_OBS_F32) {
    rc = cz_launch_obs32(t, out, reinterpret_cast<float*>(obs), n_envs, t->pipe_obs, false);
    if (rc != CZ_OK) return rc;
  } else {
    rc = cz_launch_obs64(t, out, obs, n_envs, t->pipe_obs);
    if (rc != CZ_OK) return rc;
  }
  CZ_CUDA(cudaEventRecord(t->ev_obs[nxt], t->pipe_obs));
  t->pipe_obs_pending[nxt] = 1;
  t->pipe_cur = nxt;
  t->pipe_steps += 1;
  return CZ_OK;
}

extern "C" int cz_pipeline_wait(cz_tables* t, void* stream) {
  if (!t) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (!t->pipe_ready || t->pipe_steps == 0) return CZ_OK;  // nothing enqueued since the reset (also keeps a stream capture legal)
  cudaStream_t user = (cudaStream_t)stream;
  CZ_CUDA(cudaEventRecord(t->ev_dyn, t->pipe_dyn));
  CZ_CUDA(cudaStreamWaitEvent(user, t->ev_dyn, 0));
  if (t->pipe_obs_pending[t->pipe_cur]) CZ_CUDA(cudaStreamWaitEvent(user, t->ev_obs[t->pipe_cur], 0));
  return CZ_OK;
}

extern "C" int cz_pipeline_wait_state(cz_tables* t, void* stream) {
  if (!t) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (!t->pipe_ready || t->pipe_steps == 0) return CZ_OK;
  CZ_CUDA(cudaEventRecord(t->ev_dyn, t->pipe_dyn));
  CZ_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, t->ev_dyn, 0));
  return CZ_OK;
}

extern "C" int cz_step_host(cz_tables* t, uint32_t* state_dev, const uint8_t* actions_host, double* obs_host,
                            double* reward_host, uint8_t* terminated_host, uint8_t* truncated_host, int n_envs,
                            uint32_t flags, uint64_t seed, int64_t env_offset, void* stream) {
  if (!t || !actions_host || !obs_host || !reward_host || !terminated_host || !truncated_host)
    return cz_fail(CZ_EINVAL, "%s", "null argument");
  const CzDev& T = t->dev;
  if (flags & CZ_STEP_EPISODE_STATS) {
    int rc = cz_stats_check(t, n_envs);
    if (rc != CZ_OK) return rc;
  }
  if (n_envs > t->scratch_envs) {
    if (t->d_actions) { cudaFree(t->d_actions); cudaFree(t->d_obs); cudaFree(t->d_reward); cudaFree(t->d_term); cudaFree(t->d_trunc); }
    t->scratch_envs = 0;
    size_t na = (size_t)n_envs * T.A;
    CZ_CUDA(cudaMalloc((void**)&t->d_actions, na));
    CZ_CUDA(cudaMalloc((void**)&t->d_obs, na * T.L * sizeof(double)));
    CZ_CUDA(cudaMalloc((void**)&t->d_reward, na * sizeof(double)));
    CZ_CUDA(cudaMalloc((void**)&t->d_term, na));
    CZ_CUDA(cudaMalloc((void**)&t->d_trunc, na));
    t->scratch_envs = n_envs;
  }
  cudaStream_t s = (cudaStream_t)stream;
  size_t na = (size_t)n_envs * T.A;
  CZ_CUDA(cudaMemcpyAsync(t->d_actions, actions_host, na, cudaMemcpyHostToDevice, s));
  // Large float64 batches on the specialised kernels: the step runs as column ranges and the device->host copy of range c
  // leaves on a second stream while range c + 1 is still being stepped and written, so the copy engine starts after a
  // quarter of the kernels instead of after all of them.  (The copy is > 99 % of this call: this recovers the kernels'
  // ~0.1 ms of ~11 ms, no more.)
  const int chunks = t->host_chunks;
  if (chunks > 1 && (t->simple || t->simple2) && !(flags & CZ_STEP_OBS_F32) && n_envs >= 4 * 8192) {
    int rc = cz_pipe_init(t);
    if (rc != CZ_OK) return rc;
    const bool stats = (flags & CZ_STEP_EPISODE_STATS) != 0;
    flags &= ~CZ_STEP_EPISODE_STATS;
    const int chunk = (((n_envs + chunks - 1) / chunks) + 255) & ~255;
    cudaStream_t copy = t->pipe_obs;
    int c = 0;
    for (int e0 = 0; e0 < n_envs; e0 += chunk, ++c) {
      const int n = n_envs - e0 < chunk ? n_envs - e0 : chunk;
      const size_t o = (size_t)e0 * T.A;
      rc = cz_launch<MODE_STEP>(t, state_dev + e0, state_dev + e0, true, t->d_actions + o, nullptr, nullptr, nullptr, nullptr,
                                t->d_reward + o, t->d_term + o, t->d_trunc + o, nullptr, n, flags, seed, env_offset + e0, stream,
                                n_envs);
      if (rc != CZ_OK) return rc;
      rc = cz_launch_obs64(t, state_dev + e0, t->d_obs + o * T.L, n, s, n_envs);
      if (rc != CZ_OK) return rc;
      CZ_CUDA(cudaEventRecord(t->ev_chunk[c], s));
      CZ_CUDA(cudaStreamWaitEvent(copy, t->ev_chunk[c], 0));
      CZ_CUDA(cudaMemcpyAsync(obs_host + o * T.L, t->d_obs + o * T.L, (size_t)n * T.A * T.L * sizeof(double), cudaMemcpyDeviceToHost, copy));
      CZ_CUDA(cudaMemcpyAsync(reward_host + o, t->d_reward + o, (size_t)n * T.A * sizeof(double), cudaMemcpyDeviceToHost, copy));
      CZ_CUDA(cudaMemcpyAsync(terminated_host + o, t->d_term + o, (size_t)n * T.A, cudaMemcpyDeviceToHost, copy));
      CZ_CUDA(cudaMemcpyAsync(truncated_host + o, t->d_trunc + o, (size_t)n * T.A, cudaMemcpyDeviceToHost, copy));
    }
    if (stats) {  // after every range's step; the copies do not wait for it
      rc = cz_stats_launch(t, state_dev, t->d_reward, n_envs, s);
      if (rc != CZ_OK) return rc;
    }
    CZ_CUDA(cudaEventRecord(t->ev_obs[0], copy));
    CZ_CUDA(cudaStreamWaitEvent(s, t->ev_obs[0], 0));
    CZ_CUDA(cudaStreamSynchronize(s));
    return CZ_OK;
  }
  int rc = cz_step(t, state_dev, t->d_actions, t->d_obs, t->d_reward, t->d_term, t->d_trunc, nullptr, n_envs, 1, flags, seed,
                   env_offset, 0, stream);
  if (rc != CZ_OK) return rc;
  CZ_CUDA(cudaMemcpyAsync(obs_host, t->d_obs, na * T.L * ((flags & CZ_STEP_OBS_F32) ? sizeof(float) : sizeof(double)),
                          cudaMemcpyDeviceToHost, s));
  CZ_CUDA(cudaMemcpyAsync(reward_host, t->d_reward, na * sizeof(double), cudaMemcpyDeviceToHost, s));
  CZ_CUDA(cudaMemcpyAsync(terminated_host, t->d_term, na, cudaMemcpyDeviceToHost, s));
  CZ_CUDA(cudaMemcpyAsync(truncated_host, t->d_trunc, na, cudaMemcpyDeviceToHost, s));
  CZ_CUDA(cudaStreamSynchronize(s));
  return CZ_OK;
}

#include "cz_policy.cuh"
