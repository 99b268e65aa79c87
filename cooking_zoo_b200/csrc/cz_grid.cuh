// cz_grid.cuh — the grid observation: per-cell uint8 planes of every agent's world (include/cz_b200.h, "grid observation").
//
// A pure function of the packed state, written after the dynamics like the float64 / float32 row writers, and independent of
// the observation plan.  grid u8 [n][A][C][H][W]; channel order (cz_b200.h): 7 static kinds, 5 static states, n:<Type> per
// dynamic type, chopped:<Type> / mashed:<Type> per choppable / blendable type, on_plate, then A agent groups (observer first).
//
// One warp per environment, `warps` environments per block.  The block's environments are contiguous in the output, so the
// block stages its whole byte range in shared memory at the same offset modulo 16 as in global memory: the 16-byte aligned
// middle leaves in ONE bulk store (cp.async.bulk with the L2 evict_first hint, as cz_obs_whole_kernel), the at most 15 + 15
// bytes before and after it as byte stores.  That works for any output pointer and any per-environment size (coop_test with
// two agents: 4508 bytes, not a multiple of 16).
//   1. zero the staging bytes (16-byte stores), load the environment's state column into two registers per lane;
//   2. static planes: one lane per cell reads the variant's grid byte (kind | special index << 4) and the SBITS bit;
//   3. dynamic planes: one lane per slot (D <= 32); lanes with the same (channel, cell) meet in __match_any_sync and the
//      lowest one writes the count;
//   4. agent groups: one lane per (observer, group) pair.
// Steps 2 and 3 write the observer-independent planes into all A observer copies at once.

#define GRID_WARPS 8             // environments per block (fewer when an environment's bytes are large, see cz_observe_grid)
#define GRID_SMEM_BUDGET 40960   // staging bytes per block at most (coop_test, 2 agents: 8 x 4508 = 36 KB, 6 blocks per SM)

struct CzGridDev {
  int W, H, HW, D, rows;
  int C;                      // channels
  int G0;                     // first agent channel (on_plate is G0 - 1)
  uint32_t E;                 // bytes per environment: A * C * H * W
  const uint8_t* grid;        // [V][64] static kind | special index << 4 (cz_table_desc.grid)
  const uint32_t* slot_ch;    // [D] per device slot: n channel | chopped channel << 8 | mashed channel << 16 (0: none)
};

// SUB: only the observers in `mask` (ascending) get their [C][H][W] block, M = popcount(mask) blocks per environment; block j
// is the one the full grid gives observer mask's j-th agent.  SUB = false is the full grid (mask unused).  `tid` and `bdim` are
// threadIdx.x and blockDim.x read in the kernel itself, where the compiler knows their range from the launch bounds.
template <int NA, bool SUB>
__device__ __forceinline__ void cz_grid_body(const CzGridDev& G, const uint32_t* __restrict__ state, uint8_t* __restrict__ out,
                                             int n_envs, int warps, uint32_t mask, const unsigned tid, const unsigned bdim) {
  extern __shared__ __align__(16) unsigned char gsm[];
  const unsigned full = 0xffffffffu;
  const int warp = tid >> 5, lane = tid & 31;
  const int e0 = blockIdx.x * warps;
  const int nb = n_envs - e0 < warps ? n_envs - e0 : warps;
  const int M = SUB ? __popc(mask) : NA;  // observer blocks per environment
  const uint32_t E = SUB ? (uint32_t)(M * G.C * G.HW) : G.E, bytes = (uint32_t)nb * E;
  uint8_t* gbeg = out + (size_t)e0 * E;                        // the block's bytes: [gbeg, gbeg + bytes)
  const uint32_t mis = (uint32_t)((uintptr_t)gbeg & 15u);      // gsm[mis + k] is gbeg[k]
  const uint32_t span = (mis + bytes + 15u) & ~15u;
  for (uint32_t i = tid * 16u; i < span; i += bdim * 16u) *reinterpret_cast<uint4*>(gsm + i) = make_uint4(0, 0, 0, 0);
  const int env = e0 + warp;
  const bool live = warp < nb;
  uint32_t w0 = 0, w1 = 0;  // state rows `lane` and `lane + 32` of this warp's environment (rows <= 32 + 4 + 6)
  if (live) {
    if (lane < G.rows) w0 = __ldg(state + (size_t)lane * n_envs + env);
    if (lane + 32 < G.rows) w1 = __ldg(state + (size_t)(lane + 32) * n_envs + env);
  }
  __syncthreads();
  if (live) {
    const int HW = G.HW, W = G.W, CHW = G.C * HW;
    uint8_t* b = gsm + mis + (size_t)warp * E;
    const int r_sb = G.D + NA + CZ_ROW_SBITS, r_var = G.D + NA + CZ_ROW_VARIANT;  // both >= 32 only past D + A = 32
    const uint32_t sb = r_sb < 32 ? __shfl_sync(full, w0, r_sb) : __shfl_sync(full, w1, r_sb - 32);
    const uint32_t var = r_var < 32 ? __shfl_sync(full, w0, r_var) : __shfl_sync(full, w1, r_var - 32);
    // static kinds and states
    for (int c = lane; c < HW; c += 32) {
      const int y = c / W, x = c - y * W;
      const uint32_t g = __ldg(G.grid + (size_t)var * 64 + y * 8 + x), kind = g & 15u, sp = g >> 4;
      const int k = kind >= ST_COUNTER && kind <= ST_BLOCK ? (int)kind - 1 : 0;  // Floor (and an empty cell): plane 0
      const bool s0 = (kind == ST_CUTBOARD && (sb >> sp & 1u)) || (kind == ST_BLENDER && (sb >> (4 + sp) & 1u)) ||
                      (kind == ST_SWITCH && (sb >> (12 + sp) & 1u)) || (kind == ST_BLOCK && (sb >> (16 + sp) & 1u));
      const int ks = kind == ST_CUTBOARD ? 7 : (kind == ST_BLENDER ? 8 : (kind == ST_SWITCH ? 10 : 11));
      const bool on = kind == ST_BLENDER && (sb >> (8 + sp) & 1u);
#pragma unroll
      for (int a = 0; a < NA; ++a) {
        if (SUB && a >= M) break;
        uint8_t* p = b + a * CHW + c;
        p[k * HW] = 1;
        if (s0) p[ks * HW] = 1;
        if (on) p[9 * HW] = 1;
      }
    }
    // dynamic objects: counts per (channel, cell); a key is channel * 64 + cell, ~0u for nothing
    {
      const uint32_t r = w0;  // lane s holds slot s (D <= 32)
      const bool pres = lane < G.D && (r & O_PRESENT);
      const uint32_t cell = (r & 7u) + ((r >> 3) & 7u) * (uint32_t)W;
      const uint32_t ch = pres ? __ldg(G.slot_ch + lane) : 0u;
      const uint32_t none = ~0u;
      uint32_t key[4];
      key[0] = pres ? (ch & 255u) * 64u + cell : none;
      key[1] = pres && (r & O_CHOP) && (ch >> 8 & 255u) ? (ch >> 8 & 255u) * 64u + cell : none;
      key[2] = pres && (r & O_MASH) && (ch >> 16 & 255u) ? (ch >> 16 & 255u) * 64u + cell : none;
      key[3] = pres && ((r >> 10) & 3u) == 2u ? (uint32_t)(G.G0 - 1) * 64u + cell : none;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const unsigned m = __match_any_sync(full, key[j]);
        if (key[j] != none && lane == __ffs(m) - 1) {
          const uint8_t n = (uint8_t)__popc(m);
          uint8_t* p = b + (key[j] >> 6) * HW + (key[j] & 63u);
#pragma unroll
          for (int a = 0; a < NA; ++a)
            if (!SUB || a < M) p[a * CHW] = n;
        }
      }
    }
    // agent groups: lane = observer block * NA + group; group 0 is the observer, then the other agents in ascending index
    {
      const int j = lane / NA, g = lane - j * NA;
      const int a = SUB ? (j < M ? (int)__fns(mask, 0, j + 1) : 0) : j;  // the observer of block j
      const int i = g == 0 ? a : (g <= a ? g - 1 : g);
      const int src = G.D + (i < NA ? i : 0);
      const uint32_t v0 = __shfl_sync(full, w0, src & 31), v1 = __shfl_sync(full, w1, src & 31);
      const uint32_t r = src < 32 ? v0 : v1;
      const int x = r & 7u, y = (r >> 3) & 7u, o = (r >> 6) & 7u;
      if (lane < M * NA && x < W && y < G.H) {
        uint8_t* p = b + j * CHW + (G.G0 + 7 * g) * HW + y * W + x;
        p[0] = 1;
        if (o >= 1 && o <= 4) p[o * HW] = 1;
        if (r >> 9 & 1u) p[5 * HW] = 1;
        if (r >> 15 & 1u) p[6 * HW] = 1;
      }
    }
  }
  cz_fence_async_smem();  // generic-proxy writes -> visible to the bulk copy
  __syncthreads();
  // out: the 16-byte aligned middle in one bulk store, the bytes before and after it one per thread
  const uintptr_t g0 = (uintptr_t)gbeg, g1 = g0 + bytes;
  const uintptr_t a0 = (g0 + 15u) & ~(uintptr_t)15u, a1 = g1 & ~(uintptr_t)15u;
  const uintptr_t head_end = a0 < g1 ? a0 : g1, tail_beg = a1 > head_end ? a1 : head_end;
  if (tid == 0 && a1 > a0) {
    cz_bulk_store_stream(reinterpret_cast<void*>(a0), gsm + (a0 - g0 + mis), (uint32_t)(a1 - a0));
    cz_bulk_commit();
  }
  const int t = tid;
  if (t < 16 && g0 + t < head_end) gbeg[t] = gsm[mis + t];
  if (t >= 16 && t < 32 && tail_beg + (t - 16) < g1) {
    const uintptr_t p = tail_beg + (t - 16);
    *reinterpret_cast<uint8_t*>(p) = gsm[p - g0 + mis];
  }
  if (tid == 0 && a1 > a0) cz_bulk_wait_read<0>();  // the staging bytes must outlive the read
}

template <int NA>
__global__ void __launch_bounds__(32 * GRID_WARPS)
cz_grid_kernel(const __grid_constant__ CzGridDev G, const uint32_t* __restrict__ state, uint8_t* __restrict__ out, int n_envs,
               int warps) {
  cz_grid_body<NA, false>(G, state, out, n_envs, warps, 0u, threadIdx.x, blockDim.x);
}

// The grid of the observers in `mask` only (cz_observe_grid_agents): [n][M][C][H][W]
template <int NA>
__global__ void __launch_bounds__(32 * GRID_WARPS)
cz_grid_agents_kernel(const __grid_constant__ CzGridDev G, const uint32_t* __restrict__ state, uint8_t* __restrict__ out, int n_envs,
                      int warps, uint32_t mask) {
  cz_grid_body<NA, true>(G, state, out, n_envs, warps, mask, threadIdx.x, blockDim.x);
}
