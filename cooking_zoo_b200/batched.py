"""BatchedCookingEnv — the batched entry point over N CookingZoo environments on one B200.

Keeps the reference constructor's arguments (cooking_zoo/environment/cooking_env.py:62-64:
level, meta_file, num_agents, max_steps, recipes, obs_spaces, end_condition_all_dishes,
action_scheme, reward_scheme, agent_respawn_rate, grace_period, agent_despawn_rate) and its
step/reset semantics, with every per-environment quantity becoming a leading batch axis.
This file is thin host code: tensors are torch-owned device memory, the work happens in
libcz_b200.so (include/cz_b200.h) on torch's current CUDA stream.
"""
import os
import ctypes as C

import numpy as np
import torch

from . import _native
from .tables import compile_tables, NUM_MISC, ROW_SBITS, ROW_TINFO, ROW_MARKS, ROW_VARIANT
from .grid import grid_channels


_ALWAYS_GUARD = os.environ.get("CZ_PY_DEVICE_GUARD") == "1"   # A/B: always enter torch.cuda.device(...) around library calls


class _LazyInfo:
    """Mapping view over BatchedCookingEnv.info(): nothing is decoded until a key is read."""

    def __init__(self, env):
        self._env = env

    def __getitem__(self, key):
        return self._env.info()[key]

    def keys(self):
        return ("t", "done", "recipe_done", "active", "error_flags")

    def __iter__(self):
        return iter(self.keys())

    def __len__(self):
        return 5


class BatchedCookingEnv:
    def __init__(self, num_envs, level, meta_file, num_agents, max_steps, recipes, agent_visualization=None,
                 obs_spaces=None, end_condition_all_dishes=False, action_scheme="scheme1", render=False,
                 reward_scheme=None, agent_respawn_rate=0.0, grace_period=20, agent_despawn_rate=0.0, *,
                 device="cuda:0", recipe_pool=None, layout_pool_size="auto", layout_seed=0, layouts=None,
                 auto_reset=False, seed=0, env_offset=0, pipelined=False, obs_dtype=torch.float64, stream=None,
                 pipeline_buffers=2, background_dynamics=0, background_policy=0, episode_stats=False, cook_agents=None,
                 cook_recipes=None, obs_agents=None):
        obs_spaces = obs_spaces or ["feature_vector"] * num_agents
        if obs_spaces and all(o == "grid" for o in obs_spaces):
            # per-cell u8 planes [N, A, C, H, W] written by their own kernel after the dynamics (cooking_zoo_b200.grid)
            if pipelined:
                raise NotImplementedError("the pipelined step writes feature_vector observations only")
            if obs_dtype != torch.float64:
                raise ValueError("obs_dtype applies to feature_vector observations; the grid is uint8")
            self.obs_mode = "grid"
        elif any(o != "feature_vector" for o in obs_spaces):
            raise NotImplementedError("the batched entry point builds feature_vector or grid observations, the same "
                                      "kind for every agent (symbolic/full are host object graphs in the reference)")
        else:
            self.obs_mode = "feature_vector"
        if action_scheme not in ("scheme1", "scheme3"):
            raise NotImplementedError("action_scheme must be 'scheme1' or 'scheme3' (scheme2 raises AttributeError "
                                      "in the reference itself, action_scheme2.py:15)")
        if render:
            raise NotImplementedError("rendering is out of scope")
        self.background_policy = int(background_policy)    # blocks per SM of the device cook's kernel (0: one wave)
        self.stream = stream                    # a torch.cuda.Stream every call is enqueued on (default: torch's current stream)
        self.lib = _native.load_library()       # raises when the CUDA library is missing
        if not torch.cuda.is_available():
            raise _native.NativeError("BatchedCookingEnv needs a CUDA device (there is no CPU fallback)")
        self.device = torch.device(device)
        self.num_envs, self.num_agents = int(num_envs), int(num_agents)
        self.possible_agents = ["player_" + str(r) for r in range(num_agents)]   # cooking_env.py:76
        self.tables = compile_tables(level, meta_file, num_agents, max_steps, recipes, reward_scheme,
                                     end_condition_all_dishes, grace_period, agent_respawn_rate,
                                     agent_despawn_rate, recipe_pool, layout_pool_size, layout_seed, layouts,
                                     action_scheme)
        t = self.tables
        self.obs_len, self.max_steps = t.obs_len, t.max_steps
        self.auto_reset, self.seed, self.env_offset = bool(auto_reset), int(seed), int(env_offset)
        desc, self._keep = _native.make_desc(t)
        handle = C.c_void_p()
        _native.check(self.lib.cz_tables_create(C.byref(desc), self.device.index or 0, C.byref(handle)))
        self._handle = handle
        N, A, L = self.num_envs, self.num_agents, self.obs_len
        dev = self.device
        # pipelined throughput mode: two state matrices (ping-pong), see cz_step_pipelined in cz_b200.h
        self.pipelined = bool(pipelined)
        # pipeline_buffers (2..4) state matrices; background_dynamics = blocks per SM of the dynamics kernel (0: full grid).
        # With a small grid the dynamics run behind the row writer of the previous steps (cz_pipeline_config): the
        # throughput setting for open-loop action streams, not for policies that need this step's state at once.
        self._state2 = torch.zeros((int(pipeline_buffers) if self.pipelined else 1, t.rows, N), dtype=torch.int32, device=dev)
        self.state = self._state2[0]
        if self.pipelined and (int(pipeline_buffers) != 2 or int(background_dynamics) != 0):
            _native.check(self.lib.cz_pipeline_config(self._handle, int(pipeline_buffers), int(background_dynamics)))
        # float32 observations: the float64 rows rounded element-wise (reference obs.astype(np.float32)), written
        # directly by their own kernel — half the bytes of the default
        if obs_dtype not in (torch.float64, torch.float32):
            raise ValueError("obs_dtype must be torch.float64 (the reference's dtype) or torch.float32")
        self.obs_dtype = obs_dtype
        self._flags = (_native.STEP_AUTO_RESET if self.auto_reset else 0) | \
                      (_native.STEP_OBS_F32 if obs_dtype == torch.float32 else 0)
        self.grid_channels = grid_channels(t)
        if self.lib.cz_grid_channels(self._handle) != len(self.grid_channels):
            raise _native.NativeError("libcz_b200.so and cooking_zoo_b200.grid disagree on the grid's channels")
        self._grid_shape = (N, A, len(self.grid_channels), t.height, t.width)
        # observations of the agents in obs_agents only: row / block j belongs to agent obs_agents[j] (cz_observe_agents)
        self.obs_agents = self._check_obs_agents(obs_agents)
        M = len(self.obs_agents)
        self._obs_mask = sum(1 << a for a in self.obs_agents)
        if M < A and self.pipelined:
            raise NotImplementedError("obs_agents: the pipelined step writes every agent's rows on its internal stream")
        if self.obs_mode == "grid":
            self.obs = torch.zeros((N, M) + self._grid_shape[2:], dtype=torch.uint8, device=dev)
        else:
            self.obs = torch.zeros((N, M, L), dtype=obs_dtype, device=dev)
        if self.obs_mode == "grid" or M < A:
            # dynamics without rows, then the observation writer (_writer); chosen once here, so that the methods of full
            # feature-vector rows keep their host code unchanged
            self.__class__ = _WriterEnv
        self.reward = torch.zeros((N, A), dtype=torch.float64, device=dev)
        self.terminated = torch.zeros((N, A), dtype=torch.uint8, device=dev)
        self.truncated = torch.zeros((N, A), dtype=torch.uint8, device=dev)
        self.error_flags = torch.zeros((N,), dtype=torch.int32, device=dev)
        self._actions = torch.zeros((N, A), dtype=torch.uint8, device=dev)
        self._info = _LazyInfo(self)
        self._dev_index = dev.index if dev.index is not None else torch.cuda.current_device()
        self._shape_actions = (N, A)
        self._stats = None
        if episode_stats:
            self._attach_episode_stats()
        self._cook = None
        if cook_agents is not None:
            self._attach_cook(cook_agents, cook_recipes)
        elif cook_recipes is not None:
            raise ValueError("cook_recipes applies to the agents named by cook_agents")

    def _check_obs_agents(self, obs_agents):
        """obs_agents (None: every agent) -> tuple of distinct agent indices in ascending order"""
        A = self.num_agents
        if obs_agents is None:
            return tuple(range(A))
        idx = [int(i) for i in obs_agents]
        if not idx:
            raise ValueError("obs_agents must name at least one agent")
        if len(set(idx)) != len(idx):
            raise ValueError("obs_agents must not name an agent twice")
        if any(i < 0 or i >= A for i in idx):
            raise ValueError(f"obs_agents: agent indices must lie in 0..{A - 1}")
        if idx != sorted(idx):
            raise ValueError("obs_agents must list the agents in ascending order (observation j is agent obs_agents[j])")
        return tuple(idx)

    def _attach_cook(self, cook_agents, cook_recipes):
        """agents driven by the device cook inside every step (CZ_STEP_COOK_AGENTS, cz_cook_attach)"""
        N, A, dev = self.num_envs, self.num_agents, self.device
        mask = self._cook_mask(cook_agents)
        rid = self._cook_recipe_ids(cook_recipes) if cook_recipes is not None else None
        policy = self._policy_handle()
        self._cook = {"mask": mask, "recipes": rid, "policy": policy,
                      "taken": torch.zeros((N, A), dtype=torch.uint8, device=dev), "bound": None}
        self.cook_step_crashed = torch.zeros((N,), dtype=torch.uint8, device=dev)
        self._cook_use(self._cook["taken"], 1)
        self._flags |= _native.STEP_COOK_AGENTS

    def _cook_use(self, taken, k_capacity, crashed=None):
        """attach `taken` ([k_capacity, N, A] or [N, A]) as actions_taken of the next calls; host bookkeeping only"""
        ck = self._cook
        crashed = self.cook_step_crashed if crashed is None else crashed
        key = (taken.data_ptr(), int(k_capacity), crashed.data_ptr())
        if ck["bound"] != key:
            d = _native.CookDesc()
            d.n_envs, d.k_capacity = self.num_envs, int(k_capacity)
            d.agent_mask, d.actions_taken, d.crashed = ck["mask"].data_ptr(), taken.data_ptr(), crashed.data_ptr()
            d.cook_recipes = ck["recipes"].data_ptr() if ck["recipes"] is not None else None
            _native.check(self.lib.cz_cook_attach(self._handle, ck["policy"], C.byref(d)))
            ck["bound"] = key
        self.actions_taken = taken

    def _cook_mask(self, agents):
        """cook_agents (agent indices, the same in every environment, or a bool tensor [N, A]) -> u8 bit mask [N] on the
        device"""
        N, A = self.num_envs, self.num_agents
        if isinstance(agents, torch.Tensor):
            if agents.dtype != torch.bool or tuple(agents.shape) != (N, A):
                raise ValueError("cook_agents must be a list of agent indices or a bool tensor [num_envs, num_agents]")
            bits = torch.tensor([1 << i for i in range(A)], dtype=torch.int32, device=self.device)
            return (agents.to(self.device).to(torch.int32) * bits).sum(1).to(torch.uint8).contiguous()
        idx = [int(i) for i in agents]
        if any(i < 0 or i >= A for i in idx):
            raise ValueError(f"cook_agents: agent indices must lie in 0..{A - 1}")
        m = 0
        for i in idx:
            m |= 1 << i
        return torch.full((N,), m, dtype=torch.uint8, device=self.device)

    def _cook_recipe_ids(self, cook_recipes):
        """a list of A recipe names or a [N, A] tensor of indices into tables.recipe_names -> u8 [N, A] on the device"""
        N, A = self.num_envs, self.num_agents
        if not isinstance(cook_recipes, torch.Tensor):
            names = list(cook_recipes)
            if len(names) != A or any(n not in self.tables.recipe_names for n in names):
                raise ValueError("cook_recipes must name one recipe of tables.recipe_names per agent "
                                 "(pass the names in recipe_pool)")
            cook_recipes = torch.tensor([self.tables.recipe_names.index(n) for n in names],
                                        dtype=torch.uint8).expand(N, A)
        rid = cook_recipes.to(device=self.device, dtype=torch.uint8).contiguous()
        if rid.shape != (N, A):
            raise ValueError("cook_recipes must have shape [num_envs, num_agents]")
        return rid

    def set_cook_agents(self, agents):
        """Change which agents the device cook drives (same forms as the constructor's cook_agents), e.g. between
        episodes: the mask buffer is rewritten on this environment's stream, so calls enqueued after this one see it."""
        if self._cook is None:
            raise _native.NativeError("cook agents are off: construct the environment with cook_agents=...")
        s = self.stream if self.stream is not None else torch.cuda.current_stream(self.device)
        with torch.cuda.stream(s):
            self._cook["mask"].copy_(self._cook_mask(agents))

    def _attach_episode_stats(self):
        """episode statistics on the device (cz_stats_attach): every step path updates them from here on"""
        N, A, dev = self.num_envs, self.num_agents, self.device
        st = {"return": torch.zeros((N, A), dtype=torch.float64, device=dev),
              "episode": torch.zeros((N,), dtype=torch.int32, device=dev),      # u32 bits of the EPISODE row last seen
              "open": torch.zeros((N,), dtype=torch.uint8, device=dev),
              "last_return": torch.zeros((N, A), dtype=torch.float64, device=dev),
              "last_length": torch.zeros((N,), dtype=torch.int32, device=dev),
              "last_served": torch.zeros((N,), dtype=torch.uint8, device=dev),
              "last_success": torch.zeros((N,), dtype=torch.uint8, device=dev),
              "finished": torch.zeros((N,), dtype=torch.int32, device=dev),
              "totals": torch.zeros((4 + A,), dtype=torch.float64, device=dev)}
        d = _native.StatsDesc()
        d.n_envs = N
        for field, key in (("ret", "return"), ("episode", "episode"), ("open", "open"), ("last_ret", "last_return"),
                           ("last_len", "last_length"), ("last_served", "last_served"), ("last_success", "last_success"),
                           ("finished", "finished"), ("totals", "totals")):
            setattr(d, field, st[key].data_ptr())
        with torch.cuda.device(dev):
            _native.check(self.lib.cz_stats_attach(self._handle, C.byref(d)))
        self._stats = st
        self.episode_totals_names = ["episodes", "length", "served", "success"] + \
                                    ["return:" + a for a in self.possible_agents]
        self.clear_episode_stats()
        self._flags |= _native.STEP_EPISODE_STATS

    # ------------------------------------------------------------------ helpers
    def _call(self, fn, *args):
        """one library call on this environment's device.  `with torch.cuda.device(...)` costs 20-30 us of host time per call,
        more than the two kernel launches of a step; when torch's current device already is ours (the usual case) the
        call goes straight through."""
        idx = self._dev_index
        if not _ALWAYS_GUARD and torch.cuda.current_device() == idx:
            rc = fn(*args)
        else:
            with torch.cuda.device(idx):
                rc = fn(*args)
        if rc:
            _native.check(rc)

    def _stream(self):
        if self.stream is not None:
            return C.c_void_p(self.stream.cuda_stream)
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "_policy", None):
            self.lib.cz_policy_destroy(self._policy)
            self._policy = None
        if getattr(self, "_handle", None):
            self.lib.cz_tables_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ API
    def reset(self, layout_ids=None, recipe_ids=None, mask=None):
        """reset(layout_ids[N]) -> obs[N, A, L] float64 (cooking_env.py:178-210).

        layout_ids index the compiled layout pool (default: cz_layout_draw(seed, env, 0) % P);
        recipe_ids [N, R] index tables.recipe_names; mask selects the environments to reset."""
        N = self.num_envs
        if layout_ids is None:
            lid = self.default_layout_ids(episode=0)
        else:
            if not isinstance(layout_ids, torch.Tensor) or not layout_ids.is_cuda:
                # host arrays are checked on the host; device tensors are range-checked by the kernel
                # (CZ_ERR_BAD_ID in error_flags) so that a reset never forces a device synchronisation
                chk = np.asarray(layout_ids)
                if chk.size and (chk.min() < 0 or chk.max() >= self.tables.num_layouts):
                    raise ValueError("layout id out of range")
            lid = torch.as_tensor(layout_ids, dtype=torch.int32).to(self.device).contiguous()
        if lid.shape != (N,):
            raise ValueError("layout_ids must have shape [num_envs]")
        rid = mk = None
        if recipe_ids is not None:
            if not isinstance(recipe_ids, torch.Tensor) or not recipe_ids.is_cuda:
                chk = np.asarray(recipe_ids)
                if chk.size and (chk.min() < 0 or chk.max() >= len(self.tables.recipe_names)):
                    raise ValueError("recipe_ids must be [num_envs, R] indices into tables.recipe_names")
            rid = torch.as_tensor(recipe_ids, dtype=torch.uint8).to(self.device).contiguous()
            if rid.shape != (N, self.tables.num_recipes):
                raise ValueError("recipe_ids must be [num_envs, R] indices into tables.recipe_names")
        if mask is not None:
            mk = torch.as_tensor(mask).to(torch.uint8).to(self.device).contiguous()
        with torch.cuda.device(self.device):
            f32 = self.obs_dtype == torch.float32
            written = isinstance(self, _WriterEnv)
            if self.pipelined:
                # drain the internal streams (dynamics / row writer still in flight) and keep stepping from the half
                # that holds the current state: a masked reset must land next to the untouched environments
                cur = max(0, self.lib.cz_pipeline_current(self._handle))
                _native.check(self.lib.cz_pipeline_reset(self._handle, cur))
                self.state = self._state2[cur]
            _native.check(self.lib.cz_reset(self._handle, self.state.data_ptr(), lid.data_ptr(),
                                            rid.data_ptr() if rid is not None else None,
                                            mk.data_ptr() if mk is not None else None,
                                            None if f32 or written else self.obs.data_ptr(), self.error_flags.data_ptr(),
                                            N, self._stream()))
            if written:
                self._call(*self._writer(self.obs.data_ptr(), self._stream()))
            elif f32:
                _native.check(self.lib.cz_observe_f32(self._handle, self.state.data_ptr(), self.obs.data_ptr(), N,
                                                      self._stream()))
        return self.obs

    def step(self, actions):
        """step(actions[N, A]) -> (obs f64[N,A,L], reward f64[N,A], terminated u8[N,A], truncated u8[N,A], info)
        (cooking_env.py:243-288).  Outputs are views of buffers that the next step overwrites."""
        a = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions))
        if a.shape != self._shape_actions:
            raise ValueError("actions must have shape [num_envs, num_agents]")
        if a.dtype != torch.uint8 or a.device != self.device or not a.is_contiguous():
            # staging copy on the caller's stream: in pipelined mode that stream trails the previous step's dynamics
            # (cz_step_pipelined orders it), so the buffer is never overwritten while a dynamics kernel still reads it
            self._actions.copy_(a)
            a = self._actions
        if self._cook is not None:
            self._cook_use(self._cook["taken"], 1)
        if self.pipelined:
            return self._step_pipelined(a)
        self._call(self.lib.cz_step, self._handle, self.state.data_ptr(), a.data_ptr(), self.obs.data_ptr(),
                   self.reward.data_ptr(), self.terminated.data_ptr(), self.truncated.data_ptr(),
                   self.error_flags.data_ptr(), self.num_envs, 1, self._flags, self.seed, self.env_offset, 0, self._stream())
        return self.obs, self.reward, self.terminated, self.truncated, self._info

    def step_k(self, k_steps, actions=None, action_step=0, keep_all=False):
        """k_steps consecutive steps in one call (cz_step's k_steps: one launch of the warp-per-environment kernel when
        the tables and the batch size allow it, the per-step kernels otherwise; same results either way).

        actions: uint8 [k_steps, N, A] on the device, or None: step j's actions are drawn on the device from the
        counter stream of random_actions() at step index action_step + j.  keep_all=False: the usual output buffers
        hold the LAST step's observations / rewards / flags.  keep_all=True: returns fresh [k_steps, ...] tensors with
        every step's outputs.  Not available in pipelined mode.

        With cook_agents, the cook decides for its agents before every step (their columns of `actions` are ignored)
        and actions_taken holds the applied actions: [N, A] of the last step, or a fresh [k_steps, N, A] with keep_all."""
        if self.pipelined:
            raise _native.NativeError("step_k runs on the in-place state (pipelined=False)")
        N, A, L, K = self.num_envs, self.num_agents, self.obs_len, int(k_steps)
        flags = self._flags
        a_ptr = None
        if actions is None:
            flags |= _native.STEP_DEVICE_ACTIONS
        else:
            a = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions))
            if a.shape != (K, N, A):
                raise ValueError("actions must have shape [k_steps, num_envs, num_agents]")
            a = a.to(device=self.device, dtype=torch.uint8).contiguous()
            self._k_actions = a          # keep alive until the launch has consumed it
            a_ptr = a.data_ptr()
        if self._cook is not None:
            if keep_all:
                self._cook_use(torch.empty((K, N, A), dtype=torch.uint8, device=self.device), K)
            else:
                self._cook_use(self._cook["taken"], 1)
        if keep_all:
            flags |= _native.STEP_KEEP_ALL
            obs = torch.empty((K, N, A, L), dtype=self.obs_dtype, device=self.device)
            rew = torch.empty((K, N, A), dtype=torch.float64, device=self.device)
            term = torch.empty((K, N, A), dtype=torch.uint8, device=self.device)
            trunc = torch.empty((K, N, A), dtype=torch.uint8, device=self.device)
        else:
            obs, rew, term, trunc = self.obs, self.reward, self.terminated, self.truncated
        with torch.cuda.device(self.device):
            _native.check(self.lib.cz_step(self._handle, self.state.data_ptr(), a_ptr, obs.data_ptr(), rew.data_ptr(),
                                           term.data_ptr(), trunc.data_ptr(), self.error_flags.data_ptr(), N, K, flags,
                                           self.seed, self.env_offset, int(action_step), self._stream()))
        return obs, rew, term, trunc, self._info

    def _writer(self, out, s):
        """(library function, arguments) writing the observation of grid mode or of an obs_agents subset from the current
        state into device address `out` on stream `s`"""
        h, st, N = self._handle, self.state.data_ptr(), self.num_envs
        full = self._obs_mask == (1 << self.num_agents) - 1
        if self.obs_mode == "grid":
            if full:
                return self.lib.cz_observe_grid, h, st, out, N, s
            return self.lib.cz_observe_grid_agents, h, st, self._obs_mask, out, N, s
        f32 = _native.STEP_OBS_F32 if self.obs_dtype == torch.float32 else 0
        return self.lib.cz_observe_agents, h, st, self._obs_mask, out, f32, N, s

    def _step_written(self, actions):
        """step() of grid mode and of obs_agents subsets: the dynamics (cz_step without observation rows), then the
        observation writer (_writer).  Returns (obs, reward, terminated, truncated, info); obs is u8 [N, M, C, H, W] in grid
        mode, [N, M, L] rows otherwise (M = len(obs_agents))."""
        a = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions))
        if a.shape != self._shape_actions:
            raise ValueError("actions must have shape [num_envs, num_agents]")
        if a.dtype != torch.uint8 or a.device != self.device or not a.is_contiguous():
            self._actions.copy_(a)
            a = self._actions
        if self._cook is not None:
            self._cook_use(self._cook["taken"], 1)
        s = self._stream()
        self._call(self.lib.cz_step, self._handle, self.state.data_ptr(), a.data_ptr(), None, self.reward.data_ptr(),
                   self.terminated.data_ptr(), self.truncated.data_ptr(), self.error_flags.data_ptr(), self.num_envs, 1,
                   self._flags & ~_native.STEP_OBS_F32, self.seed, self.env_offset, 0, s)
        self._call(*self._writer(self.obs.data_ptr(), s))
        return self.obs, self.reward, self.terminated, self.truncated, self._info

    def _step_k_written(self, k_steps, actions=None, action_step=0, keep_all=False):
        """step_k() of grid mode and of obs_agents subsets.  keep_all=False: one cz_step of k_steps without observation
        rows, then one observation write.  keep_all=True: k single steps, each followed by its observation write into slice
        k of a fresh [k_steps, *obs.shape] tensor."""
        N, A, K = self.num_envs, self.num_agents, int(k_steps)
        flags = self._flags & ~_native.STEP_OBS_F32      # no rows from the step itself: the writer follows
        if actions is None:
            flags |= _native.STEP_DEVICE_ACTIONS
        else:
            a = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions))
            if a.shape != (K, N, A):
                raise ValueError("actions must have shape [k_steps, num_envs, num_agents]")
            a = a.to(device=self.device, dtype=torch.uint8).contiguous()
            self._k_actions = a          # keep alive until the launch has consumed it
        s = self._stream()
        cook = self._cook is not None
        if cook:
            self._cook_use(self._cook["taken"], 1)
        with torch.cuda.device(self.device):
            if not keep_all:
                _native.check(self.lib.cz_step(self._handle, self.state.data_ptr(), None if actions is None else a.data_ptr(),
                                               None, self.reward.data_ptr(), self.terminated.data_ptr(),
                                               self.truncated.data_ptr(), self.error_flags.data_ptr(), N, K, flags, self.seed,
                                               self.env_offset, int(action_step), s))
                self._call(*self._writer(self.obs.data_ptr(), s))
                return self.obs, self.reward, self.terminated, self.truncated, self._info
            obs = torch.empty((K,) + tuple(self.obs.shape), dtype=self.obs.dtype, device=self.device)
            rew = torch.empty((K, N, A), dtype=torch.float64, device=self.device)
            term = torch.empty((K, N, A), dtype=torch.uint8, device=self.device)
            trunc = torch.empty((K, N, A), dtype=torch.uint8, device=self.device)
            if cook:   # slice j of the applied actions per single step; the raise bits ORed over the K steps
                taken = torch.empty((K, N, A), dtype=torch.uint8, device=self.device)
                crash_j = torch.empty_like(self.cook_step_crashed)
            for j in range(K):
                if cook:
                    self._cook_use(taken[j], 1, None if j == 0 else crash_j)
                _native.check(self.lib.cz_step(self._handle, self.state.data_ptr(),
                                               None if actions is None else a[j].data_ptr(), None, rew[j].data_ptr(),
                                               term[j].data_ptr(), trunc[j].data_ptr(), self.error_flags.data_ptr(), N, 1,
                                               flags, self.seed, self.env_offset, int(action_step) + j, s))
                self._call(*self._writer(obs[j].data_ptr(), s))
                if cook and j > 0:
                    with torch.cuda.stream(self.stream if self.stream is not None else torch.cuda.current_stream(self.device)):
                        self.cook_step_crashed |= crash_j
            if cook:   # the tables keep the env's own buffers attached, not the temporaries of this call
                self._cook_use(self._cook["taken"], 1)
                self.actions_taken = taken
        return obs, rew, term, trunc, self._info

    def _observe_written(self):
        with torch.cuda.device(self.device):
            self._call(*self._writer(self.obs.data_ptr(), self._stream()))
        return self.obs

    def grid_observation(self, out=None):
        """The grid observation of the current state, in either observation mode: uint8 [N, A, C, H, W] with the channels
        named by grid_channels (cooking_zoo_b200.grid; cell (x, y) at [..., y, x]).  out: a contiguous uint8 tensor of
        that shape on this device (any byte offset), or None for a new tensor."""
        if out is None:
            out = torch.empty(self._grid_shape, dtype=torch.uint8, device=self.device)
        elif (tuple(out.shape) != self._grid_shape or out.dtype != torch.uint8 or out.device != self.device
              or not out.is_contiguous()):
            raise ValueError(f"out must be a contiguous uint8 tensor of shape {self._grid_shape} on {self.device}")
        with torch.cuda.device(self.device):
            _native.check(self.lib.cz_observe_grid(self._handle, self.state.data_ptr(), out.data_ptr(), self.num_envs,
                                                   self._stream()))
        return out

    def _step_pipelined(self, a):
        self._call(self.lib.cz_step_pipelined, self._handle, self._state2.data_ptr(), a.data_ptr(), self.obs.data_ptr(),
                   self.reward.data_ptr(), self.terminated.data_ptr(), self.truncated.data_ptr(), self.error_flags.data_ptr(),
                   self.num_envs, self._flags, self.seed, self.env_offset, self._stream())
        self.state = self._state2[self.lib.cz_pipeline_current(self._handle)]
        return self.obs, self.reward, self.terminated, self.truncated, self._info

    def wait(self):
        """Pipelined mode: order everything enqueued so far before later work on torch's current stream."""
        if self.pipelined:
            with torch.cuda.device(self.device):
                _native.check(self.lib.cz_pipeline_wait(self._handle, self._stream()))

    def random_actions(self, step, out=None):
        """Uniform random actions generated on the device (the synthetic streams of BASELINE configs 3 / 4): a
        counter-based draw keyed by (seed, global environment, step, agent) -> u8 [N, A]."""
        if out is None:
            if getattr(self, "_rand_actions", None) is None:
                self._rand_actions = torch.zeros((self.num_envs, self.num_agents), dtype=torch.uint8, device=self.device)
            out = self._rand_actions
        with torch.cuda.device(self.device):
            _native.check(self.lib.cz_random_actions(self._handle, out.data_ptr(), self.num_envs, self.seed, int(step),
                                                     self.env_offset, self._stream()))
        return out

    def heuristic_actions(self, cook_recipes=None):
        """One decision of the reference's scripted cook (CookingAgent.step, cooking_agents/cooking_agent.py:9-17)
        per agent of every environment, computed on the device from the current state.

        cook_recipes: None (cook i follows recipe i of its environment), a list of A recipe names, or a
        uint8 tensor [N, A] of indices into tables.recipe_names.  Returns (actions u8 [N, A], crashed u8 [N]):
        bit i of crashed[e] is set where the reference cook would raise (its action is 0)."""
        N, A = self.num_envs, self.num_agents
        self._policy_handle()
        if getattr(self, "cook_actions", None) is None:
            self.cook_actions = torch.zeros((N, A), dtype=torch.uint8, device=self.device)
            self.cook_crashed = torch.zeros((N,), dtype=torch.uint8, device=self.device)
        rid = self._cook_recipe_ids(cook_recipes) if cook_recipes is not None else None
        with torch.cuda.device(self.device):
            if self.pipelined:     # the cook reads the state only: the observation rows may still be streaming out
                _native.check(self.lib.cz_pipeline_wait_state(self._handle, self._stream()))
            _native.check(self.lib.cz_policy_act(self._policy, self.state.data_ptr(),
                                                 rid.data_ptr() if rid is not None else None,
                                                 self.cook_actions.data_ptr(), self.cook_crashed.data_ptr(), N,
                                                 self._stream()))
        return self.cook_actions, self.cook_crashed

    def _policy_handle(self):
        """the device cook's policy (cz_policy_create), created on first use and shared by heuristic_actions and cook_agents"""
        if getattr(self, "_policy", None) is None:
            from .policy import compile_policy_tables
            desc, self._policy_keep = _native.make_policy_desc(self.tables, compile_policy_tables(self.tables))
            handle = C.c_void_p()
            _native.check(self.lib.cz_policy_create(self._handle, C.byref(desc), C.byref(handle)))
            self._policy = handle
            if self.background_policy:
                _native.check(self.lib.cz_policy_config(handle, self.background_policy))
        return self._policy

    def observe(self):
        with torch.cuda.device(self.device):
            fn = self.lib.cz_observe_f32 if self.obs_dtype == torch.float32 else self.lib.cz_observe
            _native.check(fn(self._handle, self.state.data_ptr(), self.obs.data_ptr(),
                                              self.num_envs, self._stream()))
        return self.obs

    def info(self):
        """Info tensors decoded from the packed state: t[N], done[N], recipe_done[N, R], active[N, A], error_flags[N]
        (cooking_env.py:248, 329-330).  Decoding launches small torch kernels, so step() returns a lazy
        mapping (`info["t"]`) instead of calling this on the hot path."""
        t = self.tables
        misc = self.state[t.num_dyn_slots + t.num_agents:]
        agents = self.state[t.num_dyn_slots:t.num_dyn_slots + t.num_agents]
        return {"t": misc[ROW_TINFO] & 0xFFFFF,
                "done": (misc[ROW_TINFO] >> 20) & 1,       # episode over: recipes complete or t >= max_steps
                "recipe_done": torch.stack([(misc[ROW_MARKS] >> (8 * r)) & 1 for r in range(t.num_recipes)], 1),
                "active": ((agents >> 15) & 1).T,
                "error_flags": self.error_flags}

    def default_layout_ids(self, episode=0):
        """int32 [N] on the device: pool index cz_layout_draw(seed, env_offset + e, episode) % P of every environment
        (one small kernel: the draw CZ_STEP_AUTO_RESET makes inside the step kernels)."""
        out = torch.empty((self.num_envs,), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _native.check(self.lib.cz_layout_ids(self._handle, out.data_ptr(), self.num_envs, self.seed, self.env_offset,
                                                 int(episode), self._stream()))
        return out

    # ------------------------------------------------------------------ episode statistics
    def _need_stats(self):
        if self._stats is None:
            raise _native.NativeError("episode statistics are off: construct the environment with episode_stats=True")
        return self._stats

    def episode_stats(self):
        """Per-environment episode statistics (constructor argument episode_stats=True), as views of the device buffers
        that every step updates (no copy, no synchronisation; ordered like the step's rewards and flags):
        "return" f64 [N, A] of the running episode, "last_return" f64 [N, A], "last_length" i32 [N], "last_served" u8 [N]
        (recipes whose root node is marked) and "last_success" u8 [N] (the end_condition_all_dishes condition) of the last
        finished episode, "finished" i32 [N] episodes finished since the last clear.  The rule is documented with
        CZ_STEP_EPISODE_STATS in include/cz_b200.h; a reset needs no extra call."""
        st = self._need_stats()
        return {k: st[k] for k in ("return", "last_return", "last_length", "last_served", "last_success", "finished")}

    def episode_totals(self, clear=False):
        """f64 [4 + A] device copy of the sums over every episode finished since the last clear, named by
        episode_totals_names: episodes, length, served, success, return:player_i.  The vector sharding.reduce_stats sums
        over ranks.  clear=True zeroes the accumulator on the same stream after the copy."""
        st = self._need_stats()
        s = self.stream if self.stream is not None else torch.cuda.current_stream(self.device)
        with torch.cuda.stream(s):
            out = st["totals"].clone()
            if clear:
                st["totals"].zero_()
        return out

    def clear_episode_stats(self):
        """Start a new counting window (cz_stats_clear): returns, the last-episode fields, finished and the totals become
        0; an episode that has not taken a step yet is counted whole, one already running is not counted."""
        self._need_stats()
        with torch.cuda.device(self.device):
            _native.check(self.lib.cz_stats_clear(self._handle, self.state.data_ptr(), self.num_envs, self._stream()))

    # ------------------------------------------------------------------ state import/export
    def export_state(self, env=None):
        """Canonical arrays per environment (same convention as oracle/ref_dump.dump_state)."""
        t = self.tables
        st = self.state.cpu().numpy().astype(np.uint32)
        D, A, W = t.num_dyn_slots, t.num_agents, t.width
        canon = t.canon_of_dev          # device slots are the compacted live slots (tables.py)
        envs = range(self.num_envs) if env is None else [env]
        out = []
        for e in envs:
            o = st[:D, e]
            live = np.zeros((D, 9), np.int16)
            pres = (o >> 6) & 1
            ck = (o >> 10) & 3
            cid = (o >> 12) & 31
            x, y = o & 7, (o >> 3) & 7
            live[:, 0] = pres
            live[:, 1], live[:, 2] = x, y
            live[:, 3] = (o >> 7) & 1
            live[:, 4] = ((o >> 8) & 1) * 2
            live[:, 5] = (o >> 9) & 1
            live[:, 6] = ck
            live[:, 7] = np.where(ck == 1, y * W + x, np.where(ck == 2, canon[np.minimum(cid, D - 1)], cid))
            live[:, 8] = (o >> 17) & 63
            live[pres == 0] = 0
            objs = np.zeros((t.num_canon_slots, 9), np.int16)
            objs[canon] = live
            a = st[D:D + A, e]
            agents = np.zeros((A, 6), np.int16)
            agents[:, 0], agents[:, 1], agents[:, 2] = a & 7, (a >> 3) & 7, (a >> 6) & 7
            agents[:, 3] = np.where((a >> 9) & 1, canon[np.minimum((a >> 10) & 31, D - 1)], -1)
            agents[:, 4], agents[:, 5] = (a >> 15) & 1, a >> 16
            misc = st[D + A:, e]
            sb, var = int(misc[ROW_SBITS]), int(misc[ROW_VARIANT])
            statics = np.zeros((t.num_static_slots, 4), np.int16)
            for s in range(t.num_static_slots):
                cell = int(t.static_cells[var, s])
                if cell == 0xFF:
                    continue
                g = int(t.grid[var, cell])
                kind, sp = g & 15, g >> 4
                bits = 0
                if kind == 3 and sb >> sp & 1:
                    bits |= 1
                if kind == 4:
                    bits |= (sb >> (4 + sp) & 1) | (sb >> (8 + sp) & 1) << 1
                if kind == 6:
                    bits |= (sb >> (12 + sp) & 1) << 2 | 8
                if kind == 7:
                    bits |= (sb >> (16 + sp) & 1) << 3
                statics[s] = (1, cell & 7, cell >> 3, bits)
            marks = np.array([(int(misc[ROW_MARKS]) >> (8 * r)) & 255 for r in range(t.num_recipes)], np.int32)
            out.append({"agents": agents, "objs": objs, "statics": statics, "marks": marks,
                        "t": np.int32(int(misc[ROW_TINFO]) & 0xFFFFF)})
        return out if env is None else out[0]

    def symbolic_observation(self, env):
        """The reference's "symbolic" observation (cooking_env.py:279-284: world_objects by class name plus
        "Agent") of one environment, rebuilt on the host from the device state — for debugging / rendering, not
        a hot path.  Objects are plain records: name, location, content (list of records, in content order),
        and the class's state attributes (chop_state / blend_state / free for food, status / toggle for
        appliances, orientation / holding / active for agents)."""
        from types import SimpleNamespace as Rec
        from . import entities as E
        from .policy import compile_policy_tables
        t = self.tables
        if getattr(self, "_static_lists", None) is None:
            self._static_lists = compile_policy_tables(t)
        lists, lens = self._static_lists["lists"], self._static_lists["list_len"]
        col = self.state[:, env].cpu().numpy().astype(np.uint32)
        D, A = t.num_dyn_slots, t.num_agents
        misc = col[D + A:]
        sb, var = int(misc[ROW_SBITS]), int(misc[ROW_VARIANT])
        out = {}
        by_cell = {}
        code_name = {et.static_code: n for n, et in E.ENTITY_TYPES.items() if et.kind == "static"}
        special = {E.ST_CUTBOARD: 0, E.ST_BLENDER: 1, E.ST_SWITCH: 2, E.ST_BLOCK: 3}
        for code, name in code_name.items():
            for k in range(int(lens[var, code])):
                cell = int(lists[var, code, k])
                r = Rec(name=name, location=(cell & 7, cell >> 3), content=[])
                if code in special:
                    sp = int(t.grid[var, cell]) >> 4
                    if code == E.ST_CUTBOARD:
                        r.status = "READY" if sb >> sp & 1 else "NOT_USABLE"
                    elif code == E.ST_BLENDER:
                        r.status = "READY" if sb >> (4 + sp) & 1 else "NOT_USABLE"
                        r.toggle = bool(sb >> (8 + sp) & 1)
                    elif code == E.ST_SWITCH:
                        r.switch_active = bool(sb >> (12 + sp) & 1)
                    else:
                        r.walkable = bool(sb >> (16 + sp) & 1)
                out.setdefault(name, []).append(r)
                by_cell[cell] = r
        recs = {}
        for tid, name in enumerate(t.dyn_types):
            fl = int(t.type_flags[tid])
            for s_ in range(int(t.type_base[tid]), int(t.type_base[tid]) + int(t.type_count[tid])):
                o = int(col[s_])
                if not o >> 6 & 1:
                    continue
                r = Rec(name=name, location=(o & 7, (o >> 3) & 7), content=[], free=bool(o >> 9 & 1))
                if fl & E.TF_CHOP:
                    r.chop_state = "CHOPPED" if o >> 7 & 1 else "FRESH"
                if fl & E.TF_BLEND:
                    r.blend_state = "MASHED" if o >> 8 & 1 else "FRESH"
                recs[s_] = (r, o)
                out.setdefault(name, []).append(r)
        agents = []
        for i in range(A):
            a = int(col[D + i])
            agents.append(Rec(name=f"agent-{i + 1}", location=(a & 7, (a >> 3) & 7), orientation=(a >> 6) & 7,
                              holding=recs[(a >> 10) & 31][0] if a >> 9 & 1 else None, active=bool(a >> 15 & 1)))
        out["Agent"] = agents
        for s_, (r, o) in sorted(recs.items(), key=lambda kv: (kv[1][1] >> 17) & 63):      # content order = position
            ck, cid = (o >> 10) & 3, (o >> 12) & 31
            if ck == 1:
                by_cell[(o & 63)].content.append(r)
            elif ck == 2:
                recs[cid][0].content.append(r)
        return out

    def teleport(self, env, agent, x, y):
        """Agent.move_to (world_objects.py:794-797) on one environment — test helper."""
        t = self.tables
        D = t.num_dyn_slots
        col = self.state[:, env].cpu().numpy().astype(np.uint32)
        rec = int(col[D + agent])
        xy = x | y << 3
        col[D + agent] = (rec & ~63) | xy
        if rec >> 9 & 1:
            h = (rec >> 10) & 31
            col[h] = (int(col[h]) & ~63) | xy
            for s in range(D):
                r = int(col[s])
                if r >> 6 & 1 and (r >> 10) & 3 == 2 and (r >> 12) & 31 == h:
                    col[s] = (r & ~63) | xy
        self.state[:, env] = torch.from_numpy(col.astype(np.int32)).to(self.device)


class _WriterEnv(BatchedCookingEnv):
    """A BatchedCookingEnv constructed with obs_spaces=["grid"] * num_agents or with obs_agents naming fewer than all agents:
    step / step_k / observe run the dynamics without rows, then the observation writer."""
    step = BatchedCookingEnv._step_written
    step_k = BatchedCookingEnv._step_k_written
    observe = BatchedCookingEnv._observe_written
