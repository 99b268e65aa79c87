// cz_obs_agents.cuh — observation rows of chosen observers only (cz_observe_agents, include/cz_b200.h).
//
// Row j of environment e is, element for element, row mask's j-th agent of cz_observe (float64) or cz_observe_f32 (float32):
// obs [n][M][L] with M = popcount(mask).  A step that feeds one learner among scripted partners writes 1 / A of the rows.
// Two writers, both built from the helpers of the full-row writers:
//   cz_obs_agents_kernel      packed plans (at most 64 (observer, slot) pairs, even L): the structure of cz_obs_whole_kernel —
//                             the selected rows staged whole in shared memory (table segments by cp.async, zeros over the
//                             computed range, computed slots by the lanes whose observer is selected) and ONE bulk store with
//                             the evict_first hint.  EPW = 2 stages two neighbouring environments per warp: one 2224-byte row
//                             per warp is load-latency-bound (cz_obs_single_pair_kernel), and a lone float32 row of L = 278
//                             is 1112 bytes, not a multiple of 16.
//   cz_obs_agents_any_kernel  every other plan, and outputs that are not 16-byte aligned: loops over the selected observers'
//                             (observer, slot) pairs, the rows staged whole, lane stores as wide as the output allows.
// Included by cz_kernels.cu.
#pragma once

template <typename F>
struct CzRowElt;
template <>
struct CzRowElt<double> {
  using V2 = double2;  // one table element of the lane maps (t0 / t1 count these)
  static __device__ __forceinline__ const double* table(const CzDev& T) { return T.obs_table; }
  static __device__ __forceinline__ void cp_async(V2* smem_dst, const V2* gsrc) { cz_cp_async16(smem_dst, gsrc); }
};
template <>
struct CzRowElt<float> {
  using V2 = float2;
  static __device__ __forceinline__ const float* table(const CzDev& T) { return T.obs_table32; }
  static __device__ __forceinline__ void cp_async(V2* smem_dst, const V2* gsrc) { cz_cp_async8(smem_dst, gsrc); }
};
__device__ __forceinline__ void cz_pair_put(const CzDev& T, const LaneSlot& ls, const PairRegs& p, double* span0) {
  cz_pair_store_at(T, ls, p, span0);
}
__device__ __forceinline__ void cz_pair_put(const CzDev& T, const LaneSlot& ls, const PairRegs& p, float* span0) {
  // cz_pair_store32 finds the row as stage2 + observer * L2 (then + stage_lo): hand it the stage2 that puts it at span0
  const int L2 = T.L >> 1;
  cz_pair_store32(T, ls, p, reinterpret_cast<float2*>(span0 - T.stage_lo) - ls.agent * L2, L2);
}
// the row of observer `a` among the selected ones, or -1
__device__ __forceinline__ int cz_obs_row(uint32_t mask, int a) { return (mask >> a & 1u) ? __popc(mask & ((1u << a) - 1u)) : -1; }

// The bounds of cz_obs_whole_kernel, whose structure this is: 6 blocks per SM (3 with two pairs per lane) keep the
// registers below the spill line and match what the staging block of two 2224-byte rows lets stay resident.
template <typename F, int NA, bool TWO, int EPW>
__global__ void __launch_bounds__(32 * ENVS_WARPS, (TWO ? 3 : 6) * 8 / ENVS_WARPS)
cz_obs_agents_kernel(const __grid_constant__ CzDev T, const uint32_t* __restrict__ state, F* __restrict__ obs, int n_envs,
                     uint32_t mask) {
  using V2 = typename CzRowElt<F>::V2;
  extern __shared__ __align__(16) unsigned char smem_rows[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int env0 = (blockIdx.x * ENVS_WARPS + warp) * EPW;
  if (env0 >= n_envs) return;
  const int n_here = n_envs - env0 < EPW ? n_envs - env0 : EPW;
  const int M = __popc(mask), D = T.D, tab2 = T.tab_len >> 1, L2 = T.L >> 1;
  const size_t N = (size_t)n_envs;
  V2* rows = reinterpret_cast<V2*>(smem_rows) + (size_t)warp * EPW * M * L2;

  const LaneSlot ls = cz_lane_slot_packed(T, lane);
  const int j0 = cz_obs_row(mask, ls.agent);  // the staged row of this lane's pair, -1: its observer is not selected
  LaneSlot ls1;
  int j1 = -1;
  if constexpr (TWO) {  // 33-64 (observer, slot) pairs: a lane owns pairs `lane` and `lane + 32`
    ls1 = cz_lane_slot_packed(T, lane + 32);
    j1 = cz_obs_row(mask, ls1.agent);
  }
  uint32_t var[EPW];
  PairRegs p[EPW], p1[EPW];
#pragma unroll
  for (int e = 0; e < EPW; ++e) {  // every environment's loads in flight together
    const int env = env0 + (e < n_here ? e : 0);  // a lone last environment is built twice and written once
    var[e] = __ldg(state + (size_t)(D + NA + CZ_ROW_VARIANT) * N + env);
    p[e] = cz_pair_load<NA>(T, state, N, env, var[e], ls);
    if constexpr (TWO) p1[e] = cz_pair_load<NA>(T, state, N, env, var[e], ls1);
  }
#pragma unroll
  for (int e = 0; e < EPW; ++e) {  // table segments of the selected rows: table -> their place in the staged rows
    const int env = env0 + (e < n_here ? e : 0);
    const V2* tab = reinterpret_cast<const V2*>(CzRowElt<F>::table(T)) + (size_t)var[e] * 64 * tab2 + lane;
#pragma unroll
    for (int a = 0; a < NA; ++a) {
      if (!(mask >> a & 1u)) continue;
      uint32_t cell;
      if constexpr (TWO) cell = __ldg(state + (size_t)(D + a) * N + env) & 63u;
      else cell = __shfl_sync(0xffffffffu, p[e].me, a * T.n_comp) & 63u;  // lane a * n_comp observes for agent a
      V2* row = rows + (size_t)(e * M + cz_obs_row(mask, a)) * L2;
      if (ls.t0 >= 0) CzRowElt<F>::cp_async(row + ls.t0, tab + cell * tab2);
      if (ls.t1 >= 0) CzRowElt<F>::cp_async(row + ls.t1, tab + cell * tab2 + 32);
    }
  }
  {  // never-occupied slots of the computed range are zeros
    const int n2 = T.ranges[0][1] >> 1, o2 = T.ranges[0][0] >> 1;
    V2 zero;
    zero.x = 0;
    zero.y = 0;
    for (int r = 0; r < EPW * M; ++r)
      for (int k = lane; k < n2; k += 32) rows[r * L2 + o2 + k] = zero;
  }
  __syncwarp();
#pragma unroll
  for (int e = 0; e < EPW; ++e) {
    if (j0 >= 0) cz_pair_put(T, ls, p[e], reinterpret_cast<F*>(rows + (size_t)(e * M + j0) * L2) + T.stage_lo);
    if constexpr (TWO)
      if (j1 >= 0) cz_pair_put(T, ls1, p1[e], reinterpret_cast<F*>(rows + (size_t)(e * M + j1) * L2) + T.stage_lo);
  }
  cz_cp_async_wait_all();
  cz_fence_async_smem();  // generic-proxy and cp.async writes -> visible to the async proxy
  __syncwarp();
  // the environments' rows are one contiguous block, 16-byte aligned (the host picks EPW so that it is)
  F* g = obs + (size_t)env0 * M * T.L;
  const uint32_t bytes = (uint32_t)(n_here * M * T.L) * (uint32_t)sizeof(F);
  if ((bytes & 15u) == 0) {
    if (lane == 0) {
      cz_bulk_store_stream(g, rows, bytes);
      cz_bulk_commit();
      cz_bulk_wait_read<0>();  // the staged rows must outlive the read
    }
  } else {  // a lone last environment of float32 rows whose size is not a multiple of 16 bytes
    V2* g2 = reinterpret_cast<V2*>(g);
    for (int k = lane; k < n_here * M * L2; k += 32) g2[k] = rows[k];
  }
}

// Any observation plan and any output alignment (a multiple of the element size): one warp per environment, the M rows staged
// whole (table segments, zeroed computed ranges, then the selected observers' (observer, slot) pairs in a loop over the lanes),
// copied out with the widest lane stores the output's alignment allows.
template <typename F, int NA>
__global__ void __launch_bounds__(32 * ENVS_WARPS)
cz_obs_agents_any_kernel(const __grid_constant__ CzDev T, const uint32_t* __restrict__ state, F* __restrict__ obs, int n_envs,
                         uint32_t mask, int warps_per_block) {
  extern __shared__ __align__(16) unsigned char smem_any[];
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  const int env = blockIdx.x * warps_per_block + warp;
  if (warp >= warps_per_block || env >= n_envs) return;
  const int M = __popc(mask), D = T.D, L = T.L, n_el = M * L;
  const size_t N = (size_t)n_envs;
  F* rows = reinterpret_cast<F*>(smem_any) + (size_t)warp * ((n_el + 3) & ~3);  // 16-byte aligned per warp
  const uint32_t var = __ldg(state + (size_t)(D + NA + CZ_ROW_VARIANT) * N + env);
  for (int a = 0; a < NA; ++a) {
    if (!(mask >> a & 1u)) continue;
    F* row = rows + cz_obs_row(mask, a) * L;
    const uint32_t cell = __ldg(state + (size_t)(D + a) * N + env) & 63u;
    const F* tab = CzRowElt<F>::table(T) + ((size_t)var * 64 + cell) * T.tab_len;
    for (int sg = 0; sg < T.n_segs; ++sg) {  // table segments: table -> row
      const int o = T.segs[sg][0], n = T.segs[sg][1], to = T.segs[sg][2];
      for (int k = lane; k < n; k += 32) row[o + k] = __ldg(tab + to + k);
    }
    for (int r = 0; r < T.n_ranges; ++r) {  // never-occupied slots of the computed ranges are zeros
      const int o = T.ranges[r][0], n = T.ranges[r][1];
      for (int k = lane; k < n; k += 32) row[o + k] = F(0);
    }
  }
  __syncwarp();
  // computed slots: a lane takes pairs lane, lane + 32, ... (pair = row j * n_comp + slot q)
  for (int pr = lane; pr < M * T.n_comp; pr += 32) {
    const int j = pr / T.n_comp, q = pr - j * T.n_comp;
    const LaneSlot ls = cz_lane_slot(T, q, (int)__fns(mask, 0, j + 1), lane);
    const PairRegs p = cz_pair_load<NA>(T, state, N, env, var, ls);
    cz_pair_put(T, ls, p, rows + j * L + T.stage_lo);
  }
  __syncwarp();
  F* g = obs + (size_t)env * n_el;
  const size_t bytes = (size_t)n_el * sizeof(F);
  if ((((uintptr_t)g | bytes) & 15) == 0) {
    for (int k = lane; k < (int)(bytes >> 4); k += 32) reinterpret_cast<uint4*>(g)[k] = reinterpret_cast<const uint4*>(rows)[k];
  } else if ((((uintptr_t)g | bytes) & 7) == 0) {
    for (int k = lane; k < (int)(bytes >> 3); k += 32) reinterpret_cast<uint2*>(g)[k] = reinterpret_cast<const uint2*>(rows)[k];
  } else {
    for (int k = lane; k < n_el; k += 32) g[k] = rows[k];
  }
}

#define CZ_AGENTS_INSTANCES(X, F)                                                                                              \
  X((cz_obs_agents_kernel<F, 1, false, 1>)); X((cz_obs_agents_kernel<F, 2, false, 1>)); X((cz_obs_agents_kernel<F, 3, false, 1>)); \
  X((cz_obs_agents_kernel<F, 4, false, 1>)); X((cz_obs_agents_kernel<F, 1, false, 2>)); X((cz_obs_agents_kernel<F, 2, false, 2>)); \
  X((cz_obs_agents_kernel<F, 3, false, 2>)); X((cz_obs_agents_kernel<F, 4, false, 2>)); X((cz_obs_agents_kernel<F, 1, true, 1>));  \
  X((cz_obs_agents_kernel<F, 2, true, 1>)); X((cz_obs_agents_kernel<F, 3, true, 1>)); X((cz_obs_agents_kernel<F, 4, true, 1>));    \
  X((cz_obs_agents_kernel<F, 1, true, 2>)); X((cz_obs_agents_kernel<F, 2, true, 2>)); X((cz_obs_agents_kernel<F, 3, true, 2>));    \
  X((cz_obs_agents_kernel<F, 4, true, 2>)); X((cz_obs_agents_any_kernel<F, 1>)); X((cz_obs_agents_any_kernel<F, 2>));              \
  X((cz_obs_agents_any_kernel<F, 3>)); X((cz_obs_agents_any_kernel<F, 4>))

// Rows of the observers in `mask` (validated by the caller) on `s`.  The packed writer takes 16-byte aligned outputs of packed
// plans whose staging block fits; everything else the any-plan writer.
template <typename F>
static int cz_launch_obs_agents(const cz_tables* t, const uint32_t* state, F* obs, uint32_t mask, int n_envs, cudaStream_t s) {
  const CzDev& T = t->dev;
  const int M = __builtin_popcount(mask);
  // two environments per warp where one environment's rows are a single row of float64 or at most two of float32 (a warp
  // with so little to store waits on its loads), and where one environment's float32 rows are not a multiple of 16 bytes
  const int epw = (M * (int)sizeof(F) <= 8 || (sizeof(F) == 4 && ((M * T.L) & 3) != 0)) ? 2 : 1;
  const size_t smem = (size_t)ENVS_WARPS * epw * M * T.L * sizeof(F);
  if ((t->simple || t->simple2) && ((uintptr_t)obs & 15) == 0 && smem <= t->smem_optin) {
    const int blocks = (n_envs + ENVS_WARPS * epw - 1) / (ENVS_WARPS * epw);
#define CZ_AG_GO(NA, TWO)                                                                                                      \
  if (epw == 2) cz_obs_agents_kernel<F, NA, TWO, 2><<<blocks, 32 * ENVS_WARPS, smem, s>>>(T, state, obs, n_envs, mask);         \
  else cz_obs_agents_kernel<F, NA, TWO, 1><<<blocks, 32 * ENVS_WARPS, smem, s>>>(T, state, obs, n_envs, mask)
#define CZ_AG_NA(NA) \
  if (t->simple2) { CZ_AG_GO(NA, true); } else { CZ_AG_GO(NA, false); }
    switch (T.A) {
      case 1: CZ_AG_NA(1); break;
      case 2: CZ_AG_NA(2); break;
      case 3: CZ_AG_NA(3); break;
      default: CZ_AG_NA(4); break;
    }
#undef CZ_AG_NA
#undef CZ_AG_GO
  } else {
    const size_t per_warp = (size_t)((M * T.L + 3) & ~3) * sizeof(F);
    int warps = (int)(((size_t)96 * 1024) / per_warp);  // at least two blocks per SM stay resident
    if (warps > ENVS_WARPS) warps = ENVS_WARPS;
    if (warps < 1) warps = 1;
    const size_t smem_any = per_warp * warps;
    if (smem_any > t->smem_optin) return cz_fail(CZ_ELIMIT, "%s", "observation rows too long for the row writer");
    const int blocks = (n_envs + warps - 1) / warps;
    switch (T.A) {
      case 1: cz_obs_agents_any_kernel<F, 1><<<blocks, 32 * ENVS_WARPS, smem_any, s>>>(T, state, obs, n_envs, mask, warps); break;
      case 2: cz_obs_agents_any_kernel<F, 2><<<blocks, 32 * ENVS_WARPS, smem_any, s>>>(T, state, obs, n_envs, mask, warps); break;
      case 3: cz_obs_agents_any_kernel<F, 3><<<blocks, 32 * ENVS_WARPS, smem_any, s>>>(T, state, obs, n_envs, mask, warps); break;
      default: cz_obs_agents_any_kernel<F, 4><<<blocks, 32 * ENVS_WARPS, smem_any, s>>>(T, state, obs, n_envs, mask, warps); break;
    }
  }
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}
