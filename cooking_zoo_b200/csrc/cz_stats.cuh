// cz_stats.cuh — episode statistics (CZ_STEP_EPISODE_STATS, cz_stats_attach / cz_stats_clear in cz_b200.h).
//
// The rule lives in cz_stats_rule, called by cz_stats_kernel (one thread per environment, launched after the dynamics of
// every per-step path) and by cz_warp_kernel's STATS instantiation (the record stays in registers across the K steps of
// one launch).  Included by cz_kernels.cu before cz_warp.cuh.
#pragma once

#define CZ_STATS_THREADS 256

// the attached caller-owned buffers (cz_stats_desc on the device side)
struct CzStatsDev {
  double* ret;
  uint32_t* episode;
  uint8_t* open;
  double* last_ret;
  int32_t* last_len;
  uint8_t* last_served;
  uint8_t* last_success;
  int32_t* finished;
  double* totals;
  int n;
};

// One step of one environment's record.  `seen` / `open`: the record's episode counter and open flag; `ret` / `r`: the
// running returns and this step's rewards of the NR agents the caller holds (all of them, or one per lane); `episode`,
// `tinfo`, `marks`: the post-step rows.  Returns true when the episode finished on this step; `served` / `success` then
// describe it.  The caller latches the result (cz_b200.h, rule step 3).
template <int NR>
__device__ __forceinline__ bool cz_stats_rule(uint32_t& seen, uint32_t& open, double (&ret)[NR], const double (&r)[NR],
                                              uint32_t episode, uint32_t tinfo, uint32_t marks, int R, bool end_all,
                                              uint32_t& served, uint32_t& success) {
  if (episode != seen) {  // 1. a reset since the last step (cz_reset or auto-reset): a new episode is counted
    seen = episode;
    open = 1u;
#pragma unroll
    for (int i = 0; i < NR; ++i) ret[i] = 0.0;
  }
  if (!open) return false;
#pragma unroll
  for (int i = 0; i < NR; ++i) ret[i] = __dadd_rn(ret[i], r[i]);  // 2. float64, round to nearest, step order
  if (!(tinfo & TI_DONE)) return false;
  // 3. finished: the recipes whose root node (bit 0 of MARKS byte r) is marked
  const uint32_t roots = marks & 0x01010101u & (R >= 4 ? 0xFFFFFFFFu : ((1u << (8 * R)) - 1u));
  served = (uint32_t)__popc(roots);
  success = end_all ? (served == (uint32_t)R) : (served > 0u);
  open = 0u;
  return true;
}

// Sum of a value over the block, valid in thread 0.  `red`: CZ_STATS_THREADS / 32 doubles of shared memory.
__device__ __forceinline__ double cz_stats_block_sum(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();  // `red` may still be read by the previous call
  if (lane == 0) red[warp] = v;
  __syncthreads();
  v = 0.0;
  if (threadIdx.x < CZ_STATS_THREADS / 32) v = red[threadIdx.x];
  if (warp == 0) {
#pragma unroll
    for (int o = (CZ_STATS_THREADS / 64); o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  }
  return v;
}

// The per-step record update: one thread per environment, after one step of all n_envs environments.  `misc`: the
// EPISODE..TINFO rows of the post-step state (row m at misc + m * ld); reward f64 [n][NA] of that step.  The totals are
// reduced over the block first (shuffles, then shared memory) and leave with at most one atomicAdd per field per block:
// synchronised resets with a max_steps limit finish every environment on the same step.
template <int NA>
__global__ void __launch_bounds__(CZ_STATS_THREADS)
cz_stats_kernel(const CzStatsDev S, const uint32_t* __restrict__ misc, const double* __restrict__ reward, int n_envs, int ld,
                int R, int end_all) {
  __shared__ double red[CZ_STATS_THREADS / 32];
  const int e = blockIdx.x * CZ_STATS_THREADS + threadIdx.x;
  bool fin = false;
  uint32_t len = 0, served = 0, success = 0;
  double ret[NA];
#pragma unroll
  for (int i = 0; i < NA; ++i) ret[i] = 0.0;
  if (e < n_envs) {
    const uint32_t episode = misc[(size_t)CZ_ROW_EPISODE * ld + e];
    const uint32_t tinfo = misc[(size_t)CZ_ROW_TINFO * ld + e];
    const uint32_t marks = misc[(size_t)CZ_ROW_MARKS * ld + e];
    uint32_t seen = S.episode[e], open = S.open[e];
    const uint32_t seen0 = seen, open0 = open;
    double r[NA];
#pragma unroll
    for (int i = 0; i < NA; ++i) {
      ret[i] = S.ret[(size_t)e * NA + i];
      r[i] = reward[(size_t)e * NA + i];
    }
    fin = cz_stats_rule<NA>(seen, open, ret, r, episode, tinfo, marks, R, end_all != 0, served, success);
    if (open0 || seen != seen0) {  // a closed record that saw no reset keeps every field
#pragma unroll
      for (int i = 0; i < NA; ++i) S.ret[(size_t)e * NA + i] = ret[i];
      if (seen != seen0) S.episode[e] = seen;
      if (open != open0) S.open[e] = (uint8_t)open;
    }
    if (fin) {
      len = TI_T(tinfo);
#pragma unroll
      for (int i = 0; i < NA; ++i) S.last_ret[(size_t)e * NA + i] = ret[i];
      S.last_len[e] = (int32_t)len;
      S.last_served[e] = (uint8_t)served;
      S.last_success[e] = (uint8_t)success;
      S.finished[e] += 1;
    }
  }
  if (!__syncthreads_or(fin)) return;  // the common step: nobody in this block finished
  const double v[4] = {fin ? 1.0 : 0.0, (double)len, (double)served, (double)success};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const double s = cz_stats_block_sum(v[j], red);  // integers below 2^53: exact in any order
    if (threadIdx.x == 0 && s != 0.0) atomicAdd(S.totals + j, s);
  }
#pragma unroll
  for (int i = 0; i < NA; ++i) {
    const double s = cz_stats_block_sum(fin ? ret[i] : 0.0, red);
    if (threadIdx.x == 0) atomicAdd(S.totals + 4 + i, s);
  }
}

// cz_stats_clear: a new counting window.  An environment whose episode has not taken a step (t == 0) is counted whole, one
// already running is not counted at all.
__global__ void __launch_bounds__(CZ_STATS_THREADS)
cz_stats_clear_kernel(const CzStatsDev S, const uint32_t* __restrict__ misc, int n_envs, int ld, int A) {
  const int e = blockIdx.x * CZ_STATS_THREADS + threadIdx.x;
  if (e < 4 + A) S.totals[e] = 0.0;  // n_envs >= 1: block 0 exists, and 4 + A <= 8 threads
  if (e >= n_envs) return;
  S.episode[e] = misc[(size_t)CZ_ROW_EPISODE * ld + e];
  S.open[e] = TI_T(misc[(size_t)CZ_ROW_TINFO * ld + e]) == 0u ? 1 : 0;
  for (int i = 0; i < A; ++i) {
    S.ret[(size_t)e * A + i] = 0.0;
    S.last_ret[(size_t)e * A + i] = 0.0;
  }
  S.last_len[e] = 0;
  S.last_served[e] = 0;
  S.last_success[e] = 0;
  S.finished[e] = 0;
}
