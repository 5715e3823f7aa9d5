"""RL-library facing adapters above ``MultiAgentEnv`` (SURVEY.md section 8, row f-3).

The reference's env *is* an RLlib multi-agent env when ray is installed
(gridworld/multiagent_env.py:13-20: ``class MultiAgentEnv(Env)`` with ``Env`` = RLlib's
``MultiAgentEnv`` or ``object``) and is handed to RLlib by a one-line creator
(examples/marl/rllib/heterogeneous/train.py:12-17).  ``powergridworld_b200.MultiAgentEnv`` picks
its base class the same way, so that creator works unchanged for ``num_envs == 1``.  This module
adds what a batched simulator needs on top:

* ``RLlibMultiAgentEnv``   -- the same single-env dict protocol for RLlib versions that speak the
  gymnasium API (``reset -> (obs, infos)``, ``step -> (obs, rew, terminateds, truncateds, infos)``).
* ``BatchedJointVectorEnv`` -- a gymnasium-``VectorEnv``-shaped view of a whole batch: one
  "sub-environment" per env instance, observation / action = the agents' vectors concatenated in
  the list interface's order (gridworld/multiagent_list_interface_env.py:80-111), host NumPy arrays
  in and out through the page-locked host-buffer step (``pgw_step_host``), autoreset at episode end.
* ``RLlibBatchedBaseEnv``  -- RLlib's vectorised multi-agent protocol (``BaseEnv``: ``poll`` /
  ``send_actions`` / ``try_reset`` over ``{env_id: {agent_id: value}}`` dicts) for a whole batch: RLlib
  batches policy inference over all sub-environments of a ``BaseEnv``, so one ``send_actions`` is one
  ``step_host`` of the batch.
* ``to_gym_space``          -- the package's ``Box`` / ``Dict`` stand-ins as real ``gymnasium`` (or
  ``gym``) spaces when one of them is importable.

Neither ray nor gymnasium is a dependency: the adapters are duck-typed, and inherit from the
libraries' base classes only when those import.
"""
from typing import Optional

import numpy as np

from powergridworld_b200 import spaces
from powergridworld_b200.multiagent_env import MultiAgentEnv

try:                                                   # the reference's own choice of base class
    from ray.rllib.env.multi_agent_env import MultiAgentEnv as _RllibBase
except ImportError:
    _RllibBase = object

try:
    import gymnasium as _gym
except ImportError:
    try:
        import gym as _gym
    except ImportError:
        _gym = None

_VectorBase = object
if _gym is not None and hasattr(_gym, "vector") and hasattr(_gym.vector, "VectorEnv"):
    _VectorBase = _gym.vector.VectorEnv


def _with_dtype(space, dtype):
    """``space`` with every ``Box`` in the element type ``dtype`` (the env's ``io_dtype``)."""
    if isinstance(space, dict):
        return type(space)({k: _with_dtype(v, dtype) for k, v in space.items()})
    if isinstance(space, spaces.Box) and space.dtype != dtype:
        return spaces.Box(space.low, space.high, shape=space.shape, dtype=dtype)
    return space


def to_gym_space(space):
    """``spaces.Box`` / ``spaces.Dict`` (and plain dicts of them) as gymnasium / gym spaces; the
    argument itself when neither library is installed."""
    if _gym is None:
        return space
    if isinstance(space, dict):
        return _gym.spaces.Dict({k: to_gym_space(v) for k, v in space.items()})
    if isinstance(space, spaces.Box):
        return _gym.spaces.Box(low=space.low, high=space.high, shape=space.shape, dtype=space.dtype.type)
    return space


class RLlibMultiAgentEnv(_RllibBase):
    """One env instance behind RLlib's multi-agent protocol, gymnasium flavour.

    ``config``: the scenario dict the reference's creators pass (``make_env_config(...)``),
    optionally with ``"env_cls"`` (default ``MultiAgentEnv``) and ``"device"``."""

    def __init__(self, config: dict = None, **kwargs):
        if _RllibBase is not object:
            super().__init__()
        cfg = dict(config or {}, **kwargs)
        cls = cfg.pop("env_cls", MultiAgentEnv)
        self.env = cls(**cfg)
        if self.env.num_envs != 1:
            raise ValueError("RLlib's multi-agent protocol is one env instance per object; "
                             "use BatchedJointVectorEnv for a batch")
        names = list(self.env.agent_names)
        self._agent_ids = set(names)
        self.possible_agents = names
        self.observation_spaces = {k: to_gym_space(v) for k, v in self.env.observation_space.items()}
        self.action_spaces = {k: to_gym_space(v) for k, v in self.env.action_space.items()}
        self.observation_space = to_gym_space(self.env.observation_space)
        self.action_space = to_gym_space(self.env.action_space)
        self.max_episode_steps = self.env.episode_length

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        if seed is not None:
            np.random.seed(seed)                       # the reference draws from NumPy's global RNG
        obs = self.env.reset(**(options or {}))
        return obs, {k: {} for k in obs}

    def step(self, action_dict):
        obs, rew, done, meta = self.env.step(action_dict)
        truncated = {k: False for k in done}
        infos = {k: meta[k] for k in obs if k in meta}
        common = {k: v for k, v in meta.items() if k not in self._agent_ids}
        if common:
            infos["__common__"] = common               # e.g. the shared voltage violation
        return obs, rew, done, truncated, infos

    def close(self):
        self.env.close()


class BatchedJointVectorEnv(_VectorBase):
    """All ``num_envs`` instances of a scenario as one vector env (gymnasium ``VectorEnv`` shape).

    observations ``[num_envs, obs_dim]`` and actions ``[num_envs, act_dim]`` are the agents'
    vectors concatenated in agent / component order (``agent_obs_slices`` / ``agent_act_slices``
    give each agent's columns); ``reward`` is the sum over agents (a centralised learner's
    signal), the per-agent rewards are in ``infos["agent_rewards"]`` as ``[num_agents, num_envs]``.
    All instances of a handle reach their last step together (termination is a function of the
    step count), so autoreset happens for the whole batch: the step that ends the episode returns
    the first observation of the next one and the final one under ``infos["final_observation"]``.
    Every step goes through ``step_host``: actions and results cross PCIe inside the call.
    ``io_dtype="float32"`` (passed on to the env) makes the spaces, actions and observations
    float32; rewards stay float64."""

    def __init__(self, config: dict = None, num_envs: int = 1, **kwargs):
        cfg = dict(config or {}, **kwargs)
        cls = cfg.pop("env_cls", MultiAgentEnv)
        self.env = cls(**cfg, num_envs=num_envs)
        self.num_envs = int(num_envs)
        e = self.env
        lo = np.full((e.obs_dim,), -np.inf)
        hi = np.full((e.obs_dim,), np.inf)
        alo = np.full((e.act_dim,), -np.inf)
        ahi = np.full((e.act_dim,), np.inf)
        self.agent_obs_slices, self.agent_act_slices = {}, {}
        for ag in e.agents:
            comps = getattr(ag, "envs", [ag])
            for c in comps:
                o0, on = c._slot["obs"]
                a0, an = c._slot["act"]
                lo[o0:o0 + on], hi[o0:o0 + on] = c.observation_space.low, c.observation_space.high
                alo[a0:a0 + an], ahi[a0:a0 + an] = c.action_space.low, c.action_space.high
            o0 = min(c._slot["obs"][0] for c in comps)
            a0 = min(c._slot["act"][0] for c in comps)
            self.agent_obs_slices[ag.name] = slice(o0, o0 + sum(c._slot["obs"][1] for c in comps))
            self.agent_act_slices[ag.name] = slice(a0, a0 + sum(c._slot["act"][1] for c in comps))
        dt = np.dtype(e.io_dtype)
        self.single_observation_space = to_gym_space(spaces.Box(lo, hi, dtype=dt))
        self.single_action_space = to_gym_space(spaces.Box(alo, ahi, dtype=dt))
        rep = lambda a: np.broadcast_to(a, (self.num_envs,) + a.shape).copy()
        self.observation_space = to_gym_space(spaces.Box(rep(lo), rep(hi), dtype=dt))
        self.action_space = to_gym_space(spaces.Box(rep(alo), rep(ahi), dtype=dt))
        self._act = None
        self.episodes = 0

    def reset(self, *, seed: Optional[int] = None, options: Optional[dict] = None):
        if seed is not None:
            np.random.seed(seed)
        obs = self.env.reset_host(**(options or {}))
        return np.ascontiguousarray(obs.T), {}

    def step(self, actions):
        e = self.env
        actions = np.asarray(actions, dtype=e.io_dtype)
        if actions.shape != (self.num_envs, e.act_dim):
            raise ValueError(f"actions must be [{self.num_envs}, {e.act_dim}]")
        if self._act is None:
            self._act = e._pinned()["act"]
        np.copyto(self._act.numpy(), actions.T)        # [act_dim, E], page-locked: read in place by the GPU
        obs, rew, done = e.step_host(self._act)
        obs_out = np.ascontiguousarray(obs.T)
        infos = {"agent_rewards": rew.copy()}
        terminated = done.astype(bool)
        if e._needs_reset:
            self.episodes += 1
            infos["final_observation"] = obs_out
            obs_out = np.ascontiguousarray(e.reset_host().T)
        return obs_out, rew.sum(axis=0), terminated, np.zeros(self.num_envs, dtype=bool), infos

    def close(self, **kwargs):
        self.env.close()


try:
    from ray.rllib.env.base_env import BaseEnv as _BaseEnvBase
except ImportError:
    _BaseEnvBase = object


class RLlibBatchedBaseEnv(_BaseEnvBase):
    """``num_envs`` instances behind RLlib's ``BaseEnv`` protocol (ray/rllib/env/base_env.py): env ids are
    the env indices 0 .. num_envs-1, agent ids the scenario's agent names, observations / actions the
    per-agent nested dicts of the single-env API.  ``gymnasium_api=True`` returns the six-tuple of
    ray >= 2.3 (terminateds, truncateds), else the five-tuple.  All instances of a handle end their
    episode on the same step; ``try_reset`` of the first env id resets the batch, the others collect
    their first observation from it."""

    def __init__(self, config: dict = None, num_envs: int = 1, gymnasium_api: bool = True, **kwargs):
        cfg = dict(config or {}, **kwargs)
        cls = cfg.pop("env_cls", MultiAgentEnv)
        self.env = cls(**cfg, num_envs=num_envs)
        self.num_envs = int(num_envs)
        self.gymnasium_api = bool(gymnasium_api)
        e = self.env
        dt = np.dtype(e.io_dtype)                       # the spaces of the host-buffer step's arrays
        self.observation_space = to_gym_space(_with_dtype(e.observation_space, dt))
        self.action_space = to_gym_space(_with_dtype(e.action_space, dt))
        # (agent, component or None, first row, rows) of the flat layouts
        self._obs_items, self._act_items = [], []
        for ag in e.agents:
            comps = getattr(ag, "envs", None)
            for c in (comps if comps is not None else [ag]):
                name = c.name if comps is not None else None
                self._obs_items.append((ag.name, name) + tuple(c._slot["obs"]))
                self._act_items.append((ag.name, name) + tuple(c._slot["act"]))
        self._act = None
        self._pending = None          # (obs [obs_dim, E], rew [A, E] or None, done) not yet polled
        self._reset_obs = None        # first observations of a fresh episode, handed out by try_reset
        self._reset_left = set()

    # ---- array <-> nested dict
    def _obs_of(self, obs, i):
        out = {}
        for agent, comp, o0, n in self._obs_items:
            v = obs[o0:o0 + n, i].copy()
            if comp is None:
                out[agent] = v
            else:
                out.setdefault(agent, {})[comp] = v
        return out

    def _fill_actions(self, buf, i, action):
        for agent, comp, a0, n in self._act_items:
            a = action[agent] if comp is None else action[agent][comp]
            buf[a0:a0 + n, i] = np.asarray(a, dtype=buf.dtype).reshape(n)

    # ---- BaseEnv
    def poll(self):
        e = self.env
        if self._pending is None:                         # first poll: start the episode
            self._pending = (e.reset_host(), None, False)
        obs_a, rew_a, done = self._pending
        self._pending = None
        names = e.agent_names
        obs, rew, term, trunc, infos = {}, {}, {}, {}, {}
        for i in range(self.num_envs):
            obs[i] = self._obs_of(obs_a, i)
            rew[i] = {a: (0.0 if rew_a is None else float(rew_a[k, i])) for k, a in enumerate(names)}
            term[i] = dict({a: bool(done) for a in names}, __all__=bool(done))
            trunc[i] = dict({a: False for a in names}, __all__=False)
            infos[i] = {a: {} for a in names}
        if self.gymnasium_api:
            return obs, rew, term, trunc, infos, {}
        return obs, rew, term, infos, {}

    def send_actions(self, action_dict):
        e = self.env
        if self._act is None:
            self._act = e._pinned()["act"]
        buf = self._act.numpy()
        for i, action in action_dict.items():
            self._fill_actions(buf, int(i), action)
        obs, rew, done = e.step_host(self._act)
        self._pending = (obs, rew, bool(e._needs_reset))

    def try_reset(self, env_id=None, *, seed=None, options=None):
        if seed is not None:
            np.random.seed(seed)
        if not self._reset_left:                          # first request of this episode boundary
            self._reset_obs = self.env.reset_host(**(options or {})).copy()
            self._reset_left = set(range(self.num_envs))
            self._pending = None
        ids = range(self.num_envs) if env_id is None else [int(env_id)]
        obs = {i: self._obs_of(self._reset_obs, i) for i in ids}
        self._reset_left -= set(ids)
        if self.gymnasium_api:
            return obs, {i: {a: {} for a in self.env.agent_names} for i in ids}
        return obs

    def get_sub_environments(self, as_dict: bool = False):
        return {} if as_dict else []                      # one device handle, no per-env objects

    def stop(self):
        self.env.close()
