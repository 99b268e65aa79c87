"""The reference's env wrappers re-exposed over the batched CUDA backend.

Same constructor arguments and return shapes as
  cooking_env.env                     (environment/cooking_env.py:26-43; the PettingZoo AEC surface; id cookingZooEnv-v0),
  cooking_env.parallel_env            (environment/cooking_env.py:26-46; dicts keyed "player_i"),
  environment.GymCookingEnvironment   (environment/environment.py:10-31; id cookingEnv-v1),
  multi_agent_gym.GymCookingEnvironment (environment/multi_agent_gym.py:10-34; id cookingEnvMA-v1),
backed by a BatchedCookingEnv with num_envs=1 (each call copies one small result to the host; the
batched entry point is the fast path).  gymnasium / pettingzoo are optional: when they are
importable the spaces are real gymnasium spaces and the ids get registered, otherwise light
stand-ins with the same attributes are used.
"""
from dataclasses import dataclass

import numpy as np

from .batched import BatchedCookingEnv
from .recipes import active_book

try:  # optional
    import gymnasium as _gym
except Exception:  # pragma: no cover - not installed in the build image
    _gym = None


@dataclass
class _Box:
    low: float
    high: float
    shape: tuple
    dtype: type = np.float32


@dataclass
class _Discrete:
    n: int


def _box(low, high, shape, dtype=np.float32):
    return _gym.spaces.Box(low=low, high=high, shape=shape, dtype=dtype) if _gym else _Box(low, high, shape, dtype)


def _discrete(n):
    return _gym.spaces.Discrete(n) if _gym else _Discrete(n)


class ParallelCookingEnv:
    """PettingZoo-parallel-style env: reset() -> (obs, infos); step({agent: action}) ->
    (obs, rewards, terminations, truncations, infos), all dicts keyed by "player_i"."""

    metadata = {"render_modes": [], "name": "cookingzoo_v1", "is_parallelizable": True}

    def __init__(self, level, meta_file, num_agents, max_steps, recipes, agent_visualization=None, obs_spaces=None,
                 end_condition_all_dishes=False, action_scheme="scheme1", render=False, reward_scheme=None,
                 agent_respawn_rate=0.0, grace_period=20, agent_despawn_rate=0.0, **backend_kwargs):
        if backend_kwargs.get("obs_agents") is not None:
            # the PettingZoo / gym APIs hand every agent its own observation
            raise NotImplementedError("obs_agents is not supported by the PettingZoo / gym wrappers")
        self._b = BatchedCookingEnv(1, level, meta_file, num_agents, max_steps, recipes, agent_visualization,
                                    obs_spaces, end_condition_all_dishes, action_scheme, render, reward_scheme,
                                    agent_respawn_rate, grace_period, agent_despawn_rate, **backend_kwargs)
        self.possible_agents = list(self._b.possible_agents)
        self.agents = self.possible_agents[:]
        self.recipe_names = list(recipes)
        self.max_steps = max_steps
        self._episode = 0
        self._done = True
        book = list(active_book().keys())
        # quirk C-7 (cooking_env.py:155-161): agent i's goal vector is one-hot(i) over the book
        self.goal_vectors = {a: np.eye(len(book))[i] for i, a in enumerate(self.possible_agents)}
        if self._b.obs_mode == "grid":    # per-cell u8 planes [C, H, W] of the agent's world (cooking_zoo_b200.grid)
            shape = (len(self._b.grid_channels), self._b.tables.height, self._b.tables.width)
            self.observation_spaces = {a: _box(0, 255, shape, np.uint8) for a in self.possible_agents}
        else:
            L = self._b.obs_len
            self.observation_spaces = {a: _box(-1, 1, (L,)) for a in self.possible_agents}
        self.action_spaces = {a: _discrete(self._b.tables.num_actions) for a in self.possible_agents}  # cooking_env.py:131

    def observation_space(self, agent):
        return self.observation_spaces[agent]

    def action_space(self, agent):
        return self.action_spaces[agent]

    @property
    def unwrapped(self):
        return self

    @property
    def backend(self):
        return self._b

    def reset(self, seed=None, options=None):
        """The reference re-samples the layout from the global `random` stream and ignores `seed`
        (cooking_env.py:178); here episode k takes pool layout cz_layout_index(tables, seed, env_offset, k) — for levels
        with at most 4096 initial layouts a draw from the exact distribution of the reference's parser — or
        options["layout_id"]."""
        options = options or {}
        if seed is not None:
            self._b.seed = int(seed)
        lid = options.get("layout_id")
        if lid is None:
            lid = self._b.lib.cz_layout_index(self._b._handle, self._b.seed, self._b.env_offset, self._episode)
        self._episode += 1
        obs = self._b.reset(layout_ids=np.array([lid], np.int32)).cpu().numpy()[0]
        self._obs_all = obs
        self.agents = self.possible_agents[:]
        self._done = False
        self._termination_info = ""
        self._was_active = np.ones(len(self.possible_agents), bool)
        return ({a: obs[i].copy() for i, a in enumerate(self.possible_agents)},
                {a: {} for a in self.possible_agents})

    def step(self, actions):
        """accumulated_step through the dict surface (cooking_env.py:243-269).  Only agents that are active or
        whose status changed this step appear in the returned dicts, and `self.agents` follows them: a despawned
        agent leaves (truncated=True on its despawn step, :333-350) and comes back when it respawns, while the
        episode goes on for the others; the episode ends when the recipes are complete or max_steps is reached."""
        if self._done:
            raise RuntimeError("step() called on a finished episode: call reset() first")
        A = len(self.possible_agents)
        act = np.zeros((1, A), np.uint8)
        for i, a in enumerate(self.possible_agents):
            act[0, i] = int(actions.get(a, 0))
        obs, rew, term, trunc, info = self._b.step(act)
        obs, rew = obs.cpu().numpy()[0], rew.cpu().numpy()[0]
        self._obs_all = obs
        term, trunc = term.cpu().numpy()[0].astype(bool), trunc.cpu().numpy()[0].astype(bool)
        full = self._b.info()
        t = int(full["t"][0])
        over = bool(full["done"][0])
        active = full["active"][0].cpu().numpy().astype(bool)
        done = full["recipe_done"][0].cpu().numpy().astype(bool)
        # compute_truncated sets the message only when the clock runs out (cooking_env.py:334-335); it then stays set
        if t >= self.max_steps:
            self._termination_info = f"Terminating because {self.max_steps} timesteps passed"
        relevant = active | trunc          # active, or status changed this step (despawned now / truncated by the clock)
        out_obs, out_r, out_te, out_tr, out_i = {}, {}, {}, {}, {}
        for i, a in enumerate(self.possible_agents):
            if not relevant[i]:
                continue
            out_obs[a] = obs[i].copy()
            out_r[a] = np.float64(rew[i])
            out_te[a] = bool(term[i])
            out_tr[a] = bool(trunc[i])
            out_i[a] = {"goal_vector": self.goal_vectors[a], "t": t, "termination_info": self._termination_info,
                        "recipe_done": bool(done[i]), "action": int(act[0, i]) if self._was_active[i] else 0,
                        "task": self.recipe_names[i]}
        self._was_active = active.copy()
        self.agents = [a for i, a in enumerate(self.possible_agents) if relevant[i]]     # cooking_env.py:264-266
        if over:
            self._done = True
            self.agents = []
        return out_obs, out_r, out_te, out_tr, out_i

    def render(self, **kwargs):
        raise NotImplementedError("rendering is out of scope")

    def close(self):
        self._b.close()


def parallel_env(**kwargs):
    """cooking_env.parallel_env (cooking_env.py:46)."""
    return ParallelCookingEnv(**kwargs)


class _Selector:
    """pettingzoo's agent_selector as the reference uses it (cooking_env.py:135-136, 189-190, 268): next() hands out the
    agents round-robin, is_last() says whether the agent handed out last closes the round."""

    def __init__(self, order):
        self.order, self.pos, self.selected = list(order), 0, None

    def next(self):
        self.selected = self.order[self.pos]
        self.pos = (self.pos + 1) % len(self.order)
        return self.selected

    def is_last(self):
        return self.selected == self.order[-1]


class AECCookingEnv:
    """The PettingZoo AEC surface of the reference (`cooking_env.env(...)`, cooking_env.py:26-43; AEC step :215-241):
    `agent_selection`, `last()`, one `step(action)` per selected agent; the world advances when the last agent of the
    round has stepped.  Same constructor arguments as the reference's factory.  Backed by one environment of the batched
    CUDA path; the batched entry point is the fast path, this surface is for drop-in compatibility.

    Reference behaviour kept on purpose (pinned by tests/golden/aec/aec_cfg2.npz, recorded from the reference):
    * the stepping agent's cumulative reward is NOT what gets cleared after a call: the loop variable of :228 shadows it,
      so the LAST agent of the round is cleared on every call and the others keep accumulating over the episode;
    * after an episode ends the dead-agent round cannot make progress (SURVEY.md Appendix C-8): step() on a finished
      agent raises like pettingzoo's `_was_dead_step`; call reset()."""

    metadata = {"render_modes": [], "name": "cookingzoo_v1", "is_parallelizable": True}

    def __init__(self, level, meta_file, num_agents, max_steps, recipes, agent_visualization=None, obs_spaces=None,
                 end_condition_all_dishes=False, action_scheme="scheme1", render=False, reward_scheme=None,
                 agent_respawn_rate=0.0, grace_period=20, agent_despawn_rate=0.0, **backend_kwargs):
        self._par = ParallelCookingEnv(level, meta_file, num_agents, max_steps, recipes, agent_visualization, obs_spaces,
                                       end_condition_all_dishes, action_scheme, render, reward_scheme, agent_respawn_rate,
                                       grace_period, agent_despawn_rate, **backend_kwargs)
        self.possible_agents = list(self._par.possible_agents)
        self.observation_spaces, self.action_spaces = self._par.observation_spaces, self._par.action_spaces
        self.agents = []

    def observation_space(self, agent):
        return self.observation_spaces[agent]

    def action_space(self, agent):
        return self.action_spaces[agent]

    @property
    def unwrapped(self):
        return self

    @property
    def num_agents(self):
        return len(self.agents)

    @property
    def backend(self):
        return self._par.backend

    def reset(self, seed=None, return_info=False, options=None):
        self._par.reset(seed=seed, options=options)
        self.agents = self.possible_agents[:]
        self._selector = _Selector(self.agents)
        self.agent_selection = self._selector.next()
        self.rewards = {a: 0 for a in self.agents}
        self._cumulative_rewards = {a: 0 for a in self.agents}
        self.terminations = {a: False for a in self.agents}
        self.truncations = {a: False for a in self.agents}
        self.infos = {a: {} for a in self.agents}
        self._pending = []

    def observe(self, agent):
        return self._par._obs_all[self.possible_agents.index(agent)].copy()

    def last(self, observe=True):
        a = self.agent_selection
        return (self.observe(a) if observe else None, self._cumulative_rewards[a], self.terminations[a],
                self.truncations[a], self.infos[a])

    def agent_iter(self, max_iter=2 ** 63):
        it = 0
        while self.agents and it < max_iter:
            it += 1
            yield self.agent_selection

    def step(self, action):
        if action is None:
            return          # :216-224: only meaningful right after a despawn / respawn; nothing to do otherwise (C-8)
        sel = self.agent_selection
        if self.terminations[sel] or self.truncations[sel]:
            raise ValueError("when an agent is dead, the only valid action is None")
        self._pending.append(int(action))
        for a in self.agents:
            self.rewards[a] = 0
        closing = self.agents[-1]      # what the reference's shadowed loop variable holds from here on (:228)
        if self._selector.is_last():
            acts = dict(zip(self.agents, self._pending))
            self._pending = []
            obs, rew, term, trunc, infos = self._par.step(acts)
            self.rewards, self.terminations, self.truncations, self.infos = {}, {}, {}, {}
            for a in self.possible_agents:
                if a not in rew:
                    continue
                self.rewards[a] = rew[a]
                self.terminations[a], self.truncations[a], self.infos[a] = term[a], trunc[a], infos[a]
                self._cumulative_rewards[a] = self._cumulative_rewards.get(a, 0) + rew[a]
            self.agents = [a for a in self.possible_agents if a in rew]
            self._selector = _Selector(self.agents)
            for a in self.agents:
                if self.terminations[a] or self.truncations[a]:
                    self.agent_selection = a
                    self._cumulative_rewards[closing] = 0
                    return
        self.agent_selection = self._selector.next()
        self._cumulative_rewards[closing] = 0

    def close(self):
        self._par.close()


def env(**kwargs):
    """cooking_env.env (cooking_env.py:26-43)."""
    return AECCookingEnv(**kwargs)


class GymCookingEnvironment:
    """environment.GymCookingEnvironment (environment/environment.py:5-31): single agent."""

    metadata = {"render.modes": [], "name": "cooking_zoo"}

    def __init__(self, level, meta_file, max_steps, recipes, agent_visualization=None, obs_spaces=None,
                 end_condition_all_dishes=False, action_scheme="scheme1", render=False, reward_scheme=None,
                 **backend_kwargs):
        self.zoo_env = parallel_env(level=level, meta_file=meta_file, num_agents=1, max_steps=max_steps,
                                    recipes=recipes, agent_visualization=agent_visualization, obs_spaces=obs_spaces,
                                    end_condition_all_dishes=end_condition_all_dishes, action_scheme=action_scheme,
                                    render=render, reward_scheme=reward_scheme, **backend_kwargs)
        self.observation_space = self.zoo_env.observation_space("player_0")
        self.action_space = self.zoo_env.action_space("player_0")

    def step(self, action):
        obs, reward, termination, truncation, info = self.zoo_env.step({"player_0": action})
        return obs["player_0"], reward["player_0"], termination["player_0"], truncation["player_0"], info["player_0"]

    def reset(self, **kwargs):
        obs, info = self.zoo_env.reset(**{k: v for k, v in kwargs.items() if k in ("seed", "options")})
        return obs["player_0"], info["player_0"]

    def close(self):
        self.zoo_env.close()


class GymCookingEnvironmentMA:
    """multi_agent_gym.GymCookingEnvironment (environment/multi_agent_gym.py:5-34): lists indexed by agent."""

    metadata = {"render.modes": [], "name": "multi_agent_cooking_zoo"}

    def __init__(self, level, meta_file, num_agents, max_steps, recipes, agent_visualization=None, obs_spaces=None,
                 end_condition_all_dishes=False, action_scheme="scheme1", render=False, reward_scheme=None,
                 **backend_kwargs):
        self.zoo_env = parallel_env(level=level, meta_file=meta_file, num_agents=num_agents, max_steps=max_steps,
                                    recipes=recipes, agent_visualization=agent_visualization, obs_spaces=obs_spaces,
                                    end_condition_all_dishes=end_condition_all_dishes, action_scheme=action_scheme,
                                    render=render, reward_scheme=reward_scheme, **backend_kwargs)
        self.num_agents = num_agents
        self.observation_space = self.zoo_env.observation_space("player_0")
        self.action_space = self.zoo_env.action_space("player_0")

    def step(self, actions):
        n = self.num_agents
        obs, reward, termination, truncation, info = self.zoo_env.step({f"player_{i}": actions[i] for i in range(n)})
        return ([obs[f"player_{i}"] for i in range(n)], [reward[f"player_{i}"] for i in range(n)],
                [termination[f"player_{i}"] for i in range(n)], [truncation[f"player_{i}"] for i in range(n)],
                [info[f"player_{i}"] for i in range(n)])

    def reset(self, **kwargs):
        obs, info = self.zoo_env.reset(**{k: v for k, v in kwargs.items() if k in ("seed", "options")})
        n = self.num_agents
        return [obs[f"player_{i}"] for i in range(n)], [info[f"player_{i}"] for i in range(n)]

    def close(self):
        self.zoo_env.close()


# ids of cooking_zoo/__init__.py:3-8 -> entry points here (registered with gymnasium when it is installed)
ENV_IDS = {"cookingEnv-v1": "cooking_zoo_b200.wrappers:GymCookingEnvironment",
           "cookingEnvMA-v1": "cooking_zoo_b200.wrappers:GymCookingEnvironmentMA",
           "cookingZooEnv-v0": "cooking_zoo_b200.wrappers:AECCookingEnv"}

if _gym is not None:  # pragma: no cover
    for _id, _ep in ENV_IDS.items():
        try:
            _gym.envs.registration.register(id=_id, entry_point=_ep)
        except Exception:
            pass
