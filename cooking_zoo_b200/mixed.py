"""Populations whose agent count varies per environment (BASELINE config 5).

A reference environment fixes `num_agents` at construction (cooking_env.py:62-64, 93-94), and so does
a compiled table set.  A mixed population is therefore a handful of BatchedCookingEnv groups — one per
distinct agent count, each on its own CUDA stream so their kernels overlap — behind one indexable
front.  The feature-vector length comes from the meta file, not from the agent count
(cooking_env.py:114-117), so observation rows have the same length in every group.

Stream / layout draws of environment k use the id  env_offset + (position of k in group order), where
group order lists the environments of the smallest agent count first (`stream_ids`).
"""
import numpy as np
import torch

from .batched import BatchedCookingEnv


class MixedAgentCookingEnv:
    def __init__(self, agent_counts, level, meta_file, max_steps, recipes, *, device="cuda:0", env_offset=0,
                 layouts_by_count=None, **kwargs):
        if any(o == "grid" for o in kwargs.get("obs_spaces") or ()):
            # the grid's channel count grows with the agent count: the groups would not share one observation shape
            raise NotImplementedError("MixedAgentCookingEnv builds feature_vector observations only")
        if kwargs.get("cook_agents") is not None:
            # agent indices mean different agents in groups of different sizes
            raise NotImplementedError("cook_agents is not supported by MixedAgentCookingEnv")
        if kwargs.get("obs_agents") is not None:
            # agent indices mean different agents in groups of different sizes
            raise NotImplementedError("obs_agents is not supported by MixedAgentCookingEnv")
        counts = np.asarray(agent_counts, dtype=np.int64)
        if counts.ndim != 1 or counts.size == 0 or counts.min() < 1:
            raise ValueError("agent_counts must be a non-empty vector of positive agent counts")
        if len(recipes) < counts.max():
            raise ValueError("the reference requires at least one recipe per agent")
        self.agent_counts = counts
        self.num_envs, self.max_agents = int(counts.size), int(counts.max())
        self.device = torch.device(device)
        self.groups = {}          # agent count -> BatchedCookingEnv
        self.index = {}           # agent count -> LongTensor of global environment indices
        self.streams = {}
        self.stream_ids = np.zeros(self.num_envs, np.int64)
        start = int(env_offset)
        for a in sorted(set(counts.tolist())):
            idx = np.flatnonzero(counts == a)
            kw = dict(kwargs)
            if layouts_by_count is not None:
                kw["layouts"] = layouts_by_count[a]
            self.groups[a] = BatchedCookingEnv(len(idx), level, meta_file, a, max_steps, list(recipes)[:a],
                                               device=device, env_offset=start, **kw)
            self.index[a] = torch.from_numpy(idx).to(self.device)
            self.streams[a] = torch.cuda.Stream(self.device)
            self.stream_ids[idx] = start + np.arange(len(idx))
            start += len(idx)
        self.obs_len = next(iter(self.groups.values())).obs_len
        N, A = self.num_envs, self.max_agents
        self.reward = torch.zeros((N, A), dtype=torch.float64, device=self.device)
        self.terminated = torch.zeros((N, A), dtype=torch.uint8, device=self.device)
        self.truncated = torch.zeros((N, A), dtype=torch.uint8, device=self.device)
        self.actions = torch.zeros((N, A), dtype=torch.uint8, device=self.device)

    def _fan_out(self, fn):
        """run fn(agent count, group) for every group on the group's stream, then join the caller's stream"""
        cur = torch.cuda.current_stream(self.device)
        out = {}
        for a, g in self.groups.items():
            s = self.streams[a]
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                out[a] = fn(a, g)
        for s in self.streams.values():
            cur.wait_stream(s)
        return out

    def reset(self, layout_ids=None, recipe_ids=None):
        """-> {agent count: obs f64 [n_a, a, L]}; layout_ids / recipe_ids are global [N] / [N, R_max] arrays"""
        def go(a, g):
            idx = self.index[a].cpu().numpy()
            lid = None if layout_ids is None else np.asarray(layout_ids)[idx]
            rid = None if recipe_ids is None else np.asarray(recipe_ids)[idx][:, :a]
            return g.reset(layout_ids=lid, recipe_ids=rid)
        return self._fan_out(go)

    def step(self, actions):
        """actions [N, max_agents] (columns beyond an environment's agent count are ignored) ->
        ({agent count: obs}, reward f64 [N, A_max], terminated u8, truncated u8); padded columns read 0"""
        act = torch.as_tensor(actions).to(self.device, torch.uint8)
        if act.shape != (self.num_envs, self.max_agents):
            raise ValueError("actions must have shape [num_envs, max_agents]")

        def go(a, g):
            idx = self.index[a]
            obs, rew, term, trunc, _ = g.step(act.index_select(0, idx)[:, :a].contiguous())
            self.reward[idx, :a] = rew
            self.terminated[idx, :a] = term
            self.truncated[idx, :a] = trunc
            return obs
        obs = self._fan_out(go)
        return obs, self.reward, self.terminated, self.truncated

    def cook_step(self):
        """One closed-loop step of the whole population with every action coming from the device cook: per group, on the
        group's own stream, cz_policy_act followed by the step — no gathers or scatters through the global [N, A_max]
        views, no torch kernels, two library calls per group (what BASELINE config 5 times).  Outputs stay in the groups
        (`groups[a].obs / .reward / .terminated / .truncated`); the caller's stream is joined on return."""
        self.cook_steps(1)

    def cook_steps(self, k):
        """`k` closed-loop steps of every group with ONE fork / join of the group streams around them: the groups are
        independent populations, so group a's row writer may run under group b's cook and dynamics instead of every
        phase of every group starting together (cook_step() joins the streams after each step).  The final outputs are
        those of k calls of cook_step()."""
        cur = torch.cuda.current_stream(self.device)
        for a in sorted(self.groups, reverse=True):   # the widest rows first: their writers are the longest kernels
            g, s = self.groups[a], self.streams[a]
            s.wait_stream(cur)
            g.stream = s
            try:
                for _ in range(int(k)):
                    acts, _ = g.heuristic_actions()
                    g.step(acts)
            finally:
                g.stream = None
        for s in self.streams.values():
            cur.wait_stream(s)

    def wait(self):
        """pipelined groups: order every group's observation rows before later work on the caller's stream (rewards and
        flags are ordered by step() itself: cz_step_pipelined makes the stepping stream trail the dynamics)"""
        self._fan_out(lambda a, g: g.wait())

    def heuristic_actions(self, cook_recipes=None):
        """device policy of every group -> actions u8 [N, max_agents] (padded columns 0), crashed u8 [N]"""
        crashed = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)

        def go(a, g):
            idx = self.index[a]
            cr = None if cook_recipes is None else torch.as_tensor(cook_recipes).to(self.device)[idx][:, :a]
            act, bad = g.heuristic_actions(cr)
            self.actions[idx, :a] = act
            crashed[idx] = bad
        self._fan_out(go)
        return self.actions, crashed

    def episode_stats(self):
        """episode_stats() of every group gathered into population-indexed tensors: [N, A_max] returns (padded agents
        read 0) and [N] per-environment fields.  Copies, on the caller's stream."""
        N, A = self.num_envs, self.max_agents
        out = None
        for a, g in self.groups.items():
            st = g.episode_stats()
            if out is None:
                out = {k: torch.zeros((N, A) if v.dim() == 2 else (N,), dtype=v.dtype, device=self.device)
                       for k, v in st.items()}
            idx = self.index[a]
            for k, v in st.items():
                if v.dim() == 2:
                    out[k][idx, :a] = v
                else:
                    out[k][idx] = v
        return out

    def episode_totals(self, clear=False):
        """f64 [4 + A_max]: the groups' episode_totals() summed, each padded to A_max return columns"""
        tot = torch.zeros(4 + self.max_agents, dtype=torch.float64, device=self.device)
        for a, g in self.groups.items():
            tot[:4 + a] += g.episode_totals(clear=clear)
        return tot

    def clear_episode_stats(self):
        for g in self.groups.values():
            g.clear_episode_stats()

    @property
    def episode_totals_names(self):
        return ["episodes", "length", "served", "success"] + ["return:player_" + str(i) for i in range(self.max_agents)]

    def close(self):
        for g in self.groups.values():
            g.close()
