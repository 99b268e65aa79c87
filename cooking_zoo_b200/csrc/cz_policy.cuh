// cz_policy.cuh — the reference's scripted cook as a device policy (SURVEY.md §8 f3).
//
// CookingAgent.step (cooking_agents/cooking_agent.py:9-122) + BaseAgent helpers
// (cooking_agents/base_agent.py:49-199) are a pure function of the world: the agent's private
// recipe graph is re-evaluated from scratch every call (recipe.py:77-87) and its `reachable`
// cache only memoises a property of the Floor tiles.  So the policy needs no state of its own:
// one lane reads the environment's state column (the same shared-memory columns the step kernel
// uses), evaluates every cook of that environment and writes actions u8 [n][A].
//
// Floor tiles never move, which turns both graph searches into host-built tables per static
// variant (cooking_zoo_b200/policy.py): reach[v][a] = cells b with reachable(a, b)
// (base_agent.py:94-126) and first_step[v][a][b] = walk_to_location's answer (base_agent.py:62-92,
// with its left/right/down/up expansion order and first-discoverer paths).
// The decision itself (CzPolicyDev, pol_*, pol_cook) is in cz_policy_dev.cuh.
// Included at the end of cz_kernels.cu (one translation unit, shares cz_tables / error helpers).
#pragma once

#define CZ_POLICY_THREADS 128

// Per-launch arguments of the merge instantiation (CZ_STEP_COOK_AGENTS on the per-step paths): the agents outside the
// environment's mask take the caller's action, or the draw of the counter stream at `step` (cz_random_actions).
struct CzCookStep {
  const uint8_t* agent_mask;  // [n] bit i: agent i acts by the cook
  const uint8_t* in;          // [n][A] the caller's actions, or NULL: the counter stream
  uint64_t seed, step;
  int64_t env_offset;
  int num_actions;
  int first;  // first step of the call: crashed is overwritten, later steps OR into it
};

// actions[e][i] of cz_random_actions: floor(u * len(ACTIONS)), clamped
__device__ __forceinline__ uint8_t cz_stream_action(uint64_t seed, uint64_t genv, uint64_t step, int i, int num_actions) {
  const double u = cz_uniform(seed ^ CZ_ACTION_STREAM, genv, 0, step, (uint64_t)i);
  const int a = (int)(u * num_actions);
  return (uint8_t)(a < num_actions ? a : num_actions - 1);
}

// One lane per environment; cook_recipes u8 [n][A] (book indices) or NULL = recipe i of the environment.
// MERGE = false: cz_policy_act, every agent; `M` is not read.  MERGE = true: the cook decides for the agents in M.agent_mask,
// the others are merged in from M, and `actions` is the slice the step's dynamics then read.
template <bool MERGE>
__global__ void __launch_bounds__(CZ_POLICY_THREADS)
cz_policy_kernel(const __grid_constant__ CzDev T, const __grid_constant__ CzPolicyDev P, const uint32_t* __restrict__ state,
                 const uint8_t* __restrict__ cook_recipes, uint8_t* __restrict__ actions, uint8_t* __restrict__ crashed,
                 int n_envs, const __grid_constant__ CzCookStep M) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int D = T.D, A = T.A;
  uint32_t* col = reinterpret_cast<uint32_t*>(smem_raw) + (size_t)warp * (D + A) * OSTRIDE + lane;
  uint32_t* ag = col + D * OSTRIDE;
  const size_t N = (size_t)n_envs;
  // a grid smaller than the batch (cz_policy_config: background policy of the pipelined closed loop) walks it in strides
#pragma unroll 1
  for (int env = blockIdx.x * CZ_POLICY_THREADS + threadIdx.x; env < n_envs; env += gridDim.x * CZ_POLICY_THREADS) {
  uint32_t cooks = 0xFFu;
  if constexpr (MERGE) {
    cooks = M.agent_mask[env];
    if (!cooks) {  // no cook in this environment: the state is not read
      for (int i = 0; i < A; ++i)
        actions[(size_t)env * A + i] = M.in ? M.in[(size_t)env * A + i]
                                            : cz_stream_action(M.seed, (uint64_t)(M.env_offset + env), M.step, i, M.num_actions);
      if (crashed && M.first) crashed[env] = 0;
      continue;
    }
  }
  for (int s = 0; s < D + A; ++s) cz_cp_async4(col + s * OSTRIDE, state + (size_t)s * N + env);
  const uint32_t* misc = state + (size_t)(D + A) * N;
  const uint32_t variant = misc[(size_t)CZ_ROW_VARIANT * N + env];
  const uint32_t rids = misc[(size_t)CZ_ROW_RECIPES * N + env];
  const uint32_t env_marks = misc[(size_t)CZ_ROW_MARKS * N + env];
  cz_cp_async_wait_all();
  const PolEnv pe = pol_env_masks<OSTRIDE>(T, P, col, variant);
  uint32_t bad = 0;
  for (int i = 0; i < A; ++i) {
    if (MERGE && !(cooks >> i & 1u)) {
      actions[(size_t)env * A + i] = M.in ? M.in[(size_t)env * A + i]
                                          : cz_stream_action(M.seed, (uint64_t)(M.env_offset + env), M.step, i, M.num_actions);
      continue;
    }
    // an environment scores at most CZ_MAX_RECIPES recipes; cook i follows recipe i unless told otherwise
    const uint32_t rid = cook_recipes ? cook_recipes[(size_t)env * A + i] : ((rids >> (8 * i)) & 255u);
    bool crash = false;
    uint32_t act = 0;
    // cook i follows recipe i of its environment: the environment's step has already evaluated that graph
    const uint32_t marks = (!cook_recipes && i < T.R && P.use_env_marks) ? ((env_marks >> (8 * i)) & 255u) : 0x100u;
    if (rid < (uint32_t)T.B) act = pol_cook<OSTRIDE>(T, P, pe, col, variant, ag[i * OSTRIDE], rid, marks, crash);
    else crash = true;
    if (crash) bad |= 1u << i;
    actions[(size_t)env * A + i] = (uint8_t)(crash ? 0u : act);
  }
  if (crashed) crashed[env] = (uint8_t)((MERGE && !M.first) ? (crashed[env] | bad) : bad);
  }
}

// ---- host side ---------------------------------------------------------------------------
struct cz_policy {
  const cz_tables* tables;
  int blocks_per_sm;  // 0: one thread per environment in one wave; > 0: a grid of that many blocks per SM loops over the batch
  CzPolicyDev dev;
  void* allocs[4];
  int n_allocs;
};

template <typename Tp>
static int pol_upload(cz_policy* p, const Tp* host, size_t count, const Tp** out) {
  void* d = nullptr;
  CZ_CUDA(cudaMalloc(&d, count * sizeof(Tp)));
  p->allocs[p->n_allocs++] = d;
  CZ_CUDA(cudaMemcpy(d, host, count * sizeof(Tp), cudaMemcpyHostToDevice));
  *out = (const Tp*)d;
  return CZ_OK;
}

extern "C" int cz_policy_destroy(cz_policy* p) {
  if (!p) return CZ_OK;
  cudaSetDevice(p->tables->device);
  for (int i = 0; i < p->n_allocs; ++i) cudaFree(p->allocs[i]);
  delete p;
  return CZ_OK;
}

extern "C" int cz_policy_create(const cz_tables* t, const cz_policy_desc* d, cz_policy** out) {
  if (!t || !d || !out) return cz_fail(CZ_EINVAL, "%s", "null argument");
  *out = nullptr;
  if (d->abi_version != CZ_ABI_VERSION) return cz_fail(CZ_EINVAL, "%s", "cz_policy_desc.abi_version mismatch");
  if (d->num_variants != t->dev.V) return cz_fail(CZ_EINVAL, "%s", "cz_policy_desc.num_variants differs from the tables");
  if (!d->lists || !d->list_len || !d->reach || !d->first_step) return cz_fail(CZ_EINVAL, "%s", "null policy table");
  const size_t V = (size_t)d->num_variants;
  for (size_t i = 0; i < V * 8; ++i)
    if (d->list_len[i] > CZ_MAX_CELLS) return cz_fail(CZ_ELIMIT, "%s", "static list longer than the grid");
  for (size_t i = 0; i < V * 64 * 64; ++i)
    if (d->first_step[i] > 4) return cz_fail(CZ_EINVAL, "%s", "first_step holds a non-movement action");
  CZ_CUDA(cudaSetDevice(t->device));
  cz_policy* p = new (std::nothrow) cz_policy();
  if (!p) return cz_fail(CZ_EINVAL, "%s", "out of host memory");
  p->tables = t;
  p->n_allocs = 0;
  p->blocks_per_sm = 0;
  int rc = pol_upload(p, d->lists, V * 8 * 64, &p->dev.lists);
  if (rc == CZ_OK) rc = pol_upload(p, d->list_len, V * 8, &p->dev.list_len);
  if (rc == CZ_OK) rc = pol_upload(p, d->reach, V * 64, &p->dev.reach);
  if (rc == CZ_OK) rc = pol_upload(p, d->first_step, V * 64 * 64, &p->dev.first_step);
  {
    const char* em = getenv("CZ_POLICY_ENV_MARKS");
    p->dev.use_env_marks = em ? atoi(em) : 1;
  }
  if (rc != CZ_OK) {
    cz_policy_destroy(p);
    return rc;
  }
  *out = p;
  return CZ_OK;
}

extern "C" int cz_policy_config(cz_policy* p, int blocks_per_sm) {
  if (!p || blocks_per_sm < 0 || blocks_per_sm > 16) return cz_fail(CZ_EINVAL, "%s", "cz_policy_config: 0..16 blocks per SM");
  p->blocks_per_sm = blocks_per_sm;
  return CZ_OK;
}

extern "C" int cz_policy_act(const cz_policy* p, const uint32_t* state, const uint8_t* cook_recipes, uint8_t* actions,
                             uint8_t* crashed, int n_envs, void* stream) {
  if (!p || !state || !actions) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (n_envs < 0) return cz_fail(CZ_EINVAL, "%s", "negative n_envs");
  if (n_envs == 0) return CZ_OK;
  const CzDev& T = p->tables->dev;
  const size_t smem = (size_t)(CZ_POLICY_THREADS / 32) * (T.D + T.A) * OSTRIDE * 4;
  int blocks = (n_envs + CZ_POLICY_THREADS - 1) / CZ_POLICY_THREADS;
  if (p->blocks_per_sm > 0 && blocks > p->tables->num_sms * p->blocks_per_sm) blocks = p->tables->num_sms * p->blocks_per_sm;
  // Pipelined tables in the middle of a run: the cook's kernel goes onto the library's high-priority dynamics stream, where it
  // is ordered behind the dynamics that produced `state` and gets SM slots ahead of the row writer's queued blocks (on the
  // caller's normal-priority stream it only runs once the writer of the previous step has nothing left to schedule, which
  // serialises cook and writer).  The caller's stream is ordered before and after it, as if the launch were its own.
  cz_tables* tm = const_cast<cz_tables*>(p->tables);
  const bool on_dyn = tm->policy_on_dyn && tm->pipe_ready && tm->pipe_steps > 0;
  cudaStream_t user = (cudaStream_t)stream, s = on_dyn ? tm->pipe_dyn : user;
  if (on_dyn) {
    CZ_CUDA(cudaEventRecord(tm->ev_pol_in, user));
    CZ_CUDA(cudaStreamWaitEvent(tm->pipe_dyn, tm->ev_pol_in, 0));
  }
  cz_policy_kernel<false><<<blocks, CZ_POLICY_THREADS, smem, s>>>(T, p->dev, state, cook_recipes, actions, crashed, n_envs,
                                                                 CzCookStep{});
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  if (on_dyn) {
    CZ_CUDA(cudaEventRecord(tm->ev_pol_out, tm->pipe_dyn));
    CZ_CUDA(cudaStreamWaitEvent(user, tm->ev_pol_out, 0));
  }
  return CZ_OK;
}

// ---- synthetic action streams on the device (SURVEY §8d, configs 3 and 4) -------------------------------------------

__global__ void cz_random_actions_kernel(uint8_t* __restrict__ actions, int n_envs, int A, int num_actions, uint64_t seed,
                                         uint64_t step, int64_t env_offset) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_envs * A) return;
  const int env = k / A, i = k - env * A;
  actions[k] = cz_stream_action(seed, (uint64_t)(env_offset + env), step, i, num_actions);
}

extern "C" int cz_random_actions(const cz_tables* t, uint8_t* actions, int n_envs, uint64_t seed, uint64_t step,
                                 int64_t env_offset, void* stream) {
  if (!t || !actions) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (n_envs < 0) return cz_fail(CZ_EINVAL, "%s", "negative n_envs");
  if (n_envs == 0) return CZ_OK;
  const int total = n_envs * t->dev.A, num_actions = t->dev.scheme == 1 ? 8 : 5;  // len(ACTIONS), actions.py:2-17, 39-50
  cz_random_actions_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(actions, n_envs, t->dev.A, num_actions, seed, step,
                                                                               env_offset);
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}

// ---- CZ_STEP_COOK_AGENTS (cz_cook_attach) ------------------------------------------------------------------------------
extern "C" int cz_cook_attach(cz_tables* t, const cz_policy* p, const cz_cook_desc* d) {
  if (!t) return cz_fail(CZ_EINVAL, "%s", "null argument");
  if (!d) {
    memset(&t->cook, 0, sizeof(t->cook));
    return CZ_OK;
  }
  if (!p || p->tables != t) return cz_fail(CZ_EINVAL, "%s", "cz_cook_attach: the policy must be created from these tables");
  if (d->n_envs < 1 || d->k_capacity < 1 || !d->agent_mask || !d->actions_taken)
    return cz_fail(CZ_EINVAL, "%s", "cz_cook_attach: agent_mask and actions_taken are required, n_envs and k_capacity >= 1");
  CzCookDev& C = t->cook;
  C.P = p->dev;
  C.agent_mask = d->agent_mask;
  C.cook_recipes = d->cook_recipes;
  C.actions_taken = d->actions_taken;
  C.crashed = d->crashed;
  C.k_cap = d->k_capacity;
  C.n = d->n_envs;
  return CZ_OK;
}

// the merged actions of one step of every environment of `state` into `out` [n][A] (actions_taken slice), on `s`, before
// the dynamics that read them
static int cz_cook_merge(const cz_tables* t, const uint32_t* state, const uint8_t* in, uint8_t* out, int n_envs, uint64_t seed,
                         uint64_t step, int64_t env_offset, bool first, cudaStream_t s) {
  const CzDev& T = t->dev;
  const CzCookDev& C = t->cook;
  const CzCookStep M = {C.agent_mask, in, seed, step, env_offset, T.scheme == 1 ? 8 : 5, first ? 1 : 0};
  const size_t smem = (size_t)(CZ_POLICY_THREADS / 32) * (T.D + T.A) * OSTRIDE * 4;
  const int blocks = (n_envs + CZ_POLICY_THREADS - 1) / CZ_POLICY_THREADS;
  cz_policy_kernel<true><<<blocks, CZ_POLICY_THREADS, smem, s>>>(T, C.P, state, C.cook_recipes, out, C.crashed, n_envs, M);
  g_launches.fetch_add(1);
  CZ_CUDA(cudaGetLastError());
  return CZ_OK;
}
