"""Reference-facing environment classes.

Two faces over the same CUDA step (SURVEY.md §8b):

* ``BaseEnv`` / ``SimpleEnv`` — the reference's PettingZoo ``ParallelEnv`` surface for ONE world
  (``/root/reference/src/environments/base_env.py:30-554``, ``simple_env.py:6-58``): same
  constructor, ``reset`` / ``step`` / ``state`` / spaces / ``agents`` bookkeeping, numpy dict
  outputs with the reference's dtypes, so ``driver.py`` and ``evaluate_agents`` run against it.
* ``BatchedCopsThievesEnv`` — the surface skrl's multi-agent wrapper presents to
  ``SequentialTrainer`` / ``MAPPO`` (``wrap_env(env, wrapper="pettingzoo")`` at
  ``self_play_driver.py:35``), but with ``num_envs = N``: per-agent ``(N, 180)`` float32
  observations, ``(N, 1)`` rewards / flags, ``(N, 1090)`` state, auto-reset inside the step.

Both are thin: every number comes out of ``libcat_b200.so``.
"""
from __future__ import annotations

import functools
from typing import Dict, List, Mapping, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import spaces
from .maps import Map, compile_map
from .params import EnvParams, load_physical_params
from .worlds import CatWorlds

OBJECT_TYPE_MAX = 4  # ObjectType.EMPTY (utils/object_types.py:4-9)

# The reference's BaseEnv IS a pettingzoo.ParallelEnv (base_env.py:30), and skrl's wrap_env(env, wrapper="pettingzoo")
# (self_play_driver.py:35) checks for it.  Subclass the real class wherever pettingzoo is importable; this image has
# none (SURVEY.md §8c), so the surface is duck-typed here and the base class is a plain object.
try:  # pragma: no cover - exercised only where pettingzoo exists
    from pettingzoo import ParallelEnv as _ParallelEnvBase  # type: ignore
    HAVE_PETTINGZOO = True
except Exception:
    _ParallelEnvBase = object
    HAVE_PETTINGZOO = False


def _agent_observation_space(n_rays: int, ray_length: float) -> "spaces.Dict":
    # entity.py:92-107
    return spaces.Dict({
        "distance": spaces.Box(low=0.0, high=ray_length, shape=(n_rays,), dtype=np.float16),
        "object_type": spaces.Box(low=0, high=OBJECT_TYPE_MAX, shape=(n_rays,), dtype=np.uint8),
    })


def _shared_observation_space(window: Tuple[float, float], ids: Sequence[str], n_cops: int, n_rays: int,
                              ray_length: float) -> "spaces.Dict":
    # observation_spaces.py:13-64
    max_dim = max(window)
    obs = _agent_observation_space(n_rays, ray_length)
    out = {}
    for team in (list(ids[:n_cops]), list(ids[n_cops:])):
        if not team:
            continue
        team_space = spaces.Dict({
            "own_obj_types": obs["object_type"], "own_distances": obs["distance"],
            "object_type_shared": obs["object_type"], "distance_shared": obs["distance"],
            "team_positions": spaces.Box(low=0.0, high=max_dim, shape=(len(team), 2), dtype=np.float16),
        })
        for aid in team:
            out[aid] = team_space
    return spaces.Dict(out)


class _EnvCommon:
    """Space/metadata plumbing shared by the single-world and the batched face."""

    metadata = {"render_modes": ["human", "rgb_array"]}  # base_env.py:49

    def _setup_common(self, map: Map, cmap, params: EnvParams, window: Optional[Tuple[float, float]] = None) -> None:
        self.map = map
        self.width, self.height = map.window_dimensions
        self.possible_agents: List[str] = cmap.agent_ids                     # base_env.py:96
        self._agent_index = {a: i for i, a in enumerate(self.possible_agents)}
        obs_space = _agent_observation_space(params.n_rays, params.ray_length)
        self.observation_spaces = {a: obs_space for a in self.possible_agents}  # base_env.py:102-105
        self.action_spaces = {a: spaces.Discrete(4) for a in self.possible_agents}  # entity.py:88-90
        shared = _shared_observation_space(window or map.window_dimensions, self.possible_agents, cmap.n_cops,
                                           params.n_rays, params.ray_length)
        self.shared_observation_spaces = shared                              # base_env.py:113-115
        self._shared_observation_spaces = shared
        self.state_space = shared

    def observation_space(self, agent: str):
        return self.observation_spaces[agent]

    def action_space(self, agent: str):
        return self.action_spaces[agent]

    def get_base_observation_space_structure(self):  # base_env.py:243-253
        return self._shared_observation_spaces

    @functools.lru_cache(maxsize=None)
    def get_nested_agent_observation_spaces(self):  # base_env.py:256-284
        flat = {}
        for aid in self._shared_observation_spaces:
            sp = dict(self._shared_observation_spaces[aid].spaces.items())
            for other in self._shared_observation_spaces:
                if other != aid:
                    for key, s in self._shared_observation_spaces[other].spaces.items():
                        sp[f"{other}_{key}"] = s
            flat[aid] = spaces.Dict(sp)
        return spaces.Dict(flat)


def split_worlds(num_envs: int, n_maps: int) -> List[int]:
    """``num_envs`` worlds over ``n_maps`` maps as evenly as possible, the remainder to the first maps."""
    num_envs, n_maps = int(num_envs), int(n_maps)
    if n_maps < 1 or num_envs < n_maps:
        raise ValueError(f"cannot split {num_envs} worlds over {n_maps} maps (at least one world per map)")
    q, r = divmod(num_envs, n_maps)
    return [q + (1 if m < r else 0) for m in range(n_maps)]


def _make_params(max_step_count: int, time_step: float, physical: Optional[dict], **over) -> EnvParams:
    phys = dict(load_physical_params()) if physical is None else dict(physical)
    p = EnvParams(dt=float(time_step), max_step_count=int(max_step_count), **phys)
    for k, v in over.items():
        setattr(p, k, v)
    return p


class BaseEnv(_EnvCommon, _ParallelEnvBase):
    """Single-world PettingZoo ``ParallelEnv`` face (``base_env.py:30``): a real ``pettingzoo.ParallelEnv`` subclass
    when pettingzoo is importable (``HAVE_PETTINGZOO``), the same surface duck-typed otherwise.  Needs a CUDA device."""

    def __init__(self, map: Map, map_image=None, render_mode=None, max_step_count: int = 400,
                 time_step: float = 1 / 15.0, *, device: Union[str, torch.device] = "cuda:0",
                 physical_params: Optional[dict] = None, stale_shape_cache: bool = True):
        assert render_mode is None or render_mode in self.metadata["render_modes"]  # base_env.py:117
        self.render_mode = render_mode
        self.map_image = map_image
        self.max_step_count = max_step_count
        self.time_step = time_step
        self.step_count = 0
        params = _make_params(max_step_count, time_step, physical_params, auto_reset=0,
                              stale_shape_cache=int(stale_shape_cache))
        self._cmap = compile_map(map)
        self._params = params
        self._setup_common(map, self._cmap, params)
        # One world, consumed on the CPU every step: every output lives in mapped pinned host memory, so a step
        # is one kernel launch + one stream synchronisation, and the dicts below are built from numpy views.
        self._w = CatWorlds(self._cmap, 1, device=device, params=params, want_f32=False, want_shared=True,
                            pinned_outputs=True)
        self._acts = torch.zeros((1, len(self.possible_agents)), dtype=torch.uint8).pin_memory()
        self._acts_np = self._acts.numpy()
        w = self._w
        self._np = {k: getattr(w, k).numpy() for k in ("obs_dist", "obs_type", "reward", "terminated", "truncated",
                                                         "winner", "shared_dist", "shared_type", "team_pos")}
        self.agents: List[str] = []
        self._np_random_seed = None

    # ------------------------------------------------------------------ helpers
    def _observations(self) -> Dict[str, dict]:
        d, t = self._np["obs_dist"][0], self._np["obs_type"][0]
        return {a: {"distance": d[i].copy(), "object_type": t[i].copy()} for i, a in enumerate(self.possible_agents)}

    def _shared(self, obs: Dict[str, dict]) -> Dict[str, dict]:
        # observation_spaces.py:123-129 — team-mates share (alias) the merged arrays
        sd = self._np["shared_dist"][0].copy()
        st = self._np["shared_type"][0].copy()
        tp = self._np["team_pos"][0].copy()
        nc, na = self._cmap.n_cops, len(self.possible_agents)
        team_sd, team_st = [sd[0], sd[1]], [st[0], st[1]]      # one array object per team, shared by its members
        team_tp = [tp[0:nc], tp[nc:na]]
        out = {}
        for i, a in enumerate(self.possible_agents):
            team = 0 if i < nc else 1
            out[a] = {"own_obj_types": obs[a]["object_type"], "own_distances": obs[a]["distance"],
                      "object_type_shared": team_st[team], "distance_shared": team_sd[team],
                      "team_positions": team_tp[team]}
        return out

    # ------------------------------------------------------------------ PettingZoo API
    def reset(self, seed: Optional[int] = None, options: Optional[dict] = None):  # base_env.py:286-352
        if seed is not None:
            # base_env.py:307-311 re-creates np_random, so reset(seed=s) reproduces the same spawn every time:
            # re-key Philox AND restart the episode counter that is part of its key
            self._np_random_seed = seed
            self._w.set_seed(seed, restart_episodes=True)
        self.agents = self.possible_agents[:]
        self._w.reset()
        self._w.synchronize()
        observations = self._observations()
        infos = {a: {} for a in self.agents}
        self._state = self._shared(observations)
        self.step_count = 0
        return observations, infos

    def step(self, action: Mapping[str, int]):  # base_env.py:354-413
        self.step_count += 1
        if not action:
            self.agents = []
            return {}, {}, {}, {}, {}
        for i, a in enumerate(self.possible_agents):
            self._acts_np[0, i] = int(action[a])
        self._w.step(self._acts)
        self._w.synchronize()
        observations = self._observations()
        rew = self._np["reward"][0]
        terminated = bool(self._np["terminated"][0])
        truncated = bool(self._np["truncated"][0])
        winner_code = int(self._np["winner"][0])
        agents = self.agents
        rewards = {a: float(rew[self._agent_index[a]]) for a in agents}
        terminations = {a: terminated for a in agents}
        truncations = {a: truncated for a in agents}
        self._state = self._shared(observations)
        winner = None
        if terminated:
            self.agents = []
            winner = "cop" if winner_code == 0 else "thief"
        infos = {a: {"winner": winner} for a in agents}
        return {a: observations[a] for a in agents}, rewards, terminations, truncations, infos

    def state(self) -> dict:  # base_env.py:415-425
        return self._state

    def render(self):
        """``rgb_array``: the world drawn on the GPU, ``render.render_rgb`` bit for bit (numpy (W, H, 3) uint8)."""
        if self.render_mode == "rgb_array":
            return self._w.render_frames()[0].cpu().numpy()
        return None

    def close(self):
        self._w.close()

    def _get_info(self):  # base_env.py:459-475
        return {"step_count": self.step_count, "thief_count": self._cmap.n_thieves, "cop_count": self._cmap.n_cops}


class SimpleEnv(BaseEnv):
    """``simple_env.py:6-58``: the class every reference driver instantiates (dt 1/60, rgb_array)."""

    def __init__(self, map: Map, render_mode="rgb_array", map_image=None, max_step_count: int = 400,
                 time_step: float = 1 / 60.0, **kw):
        super().__init__(map=map, map_image=map_image, render_mode=render_mode, max_step_count=max_step_count,
                         time_step=time_step, **kw)

    def _get_info(self):
        info = super()._get_info()
        pos = self._w.get_state()["pos"][0].cpu().numpy()
        nc = self._cmap.n_cops
        info.update({"environment_type": "SimpleEnv",
                     "thief_positions": [tuple(int(v) for v in p) for p in pos[nc:]],
                     "cop_positions": [tuple(int(v) for v in p) for p in pos[:nc]]})
        return info


class BatchedCopsThievesEnv(_EnvCommon, _ParallelEnvBase):
    """N worlds behind the surface skrl's multi-agent trainers use (SURVEY.md §8b, Appendix D).

    ``agents`` never empties: finished worlds are re-spawned inside the step kernel and report the
    observation of the new episode (SURVEY.md C-10), with the terminal reward / flags of the old one.

    ``final_observations=True``: the step kernel also keeps the last observation of every episode that ends, the
    gymnasium ``final_observation``: ``infos[agent]["final_observation"]`` is an (N, 2R) view of that agent's final
    observation, and ``final_state()`` / ``final_critic()`` the final ``state()`` / ``critic()``.  They are written
    only for the worlds that end in the step and are valid where ``terminated``; a truncated (timed-out) episode can be
    bootstrapped from them (``MAPPOConfig.time_limit_bootstrap``).

    Mixed maps: ``map`` may be a sequence of maps (at most 8, all with the same cops and thieves).  ``num_envs`` is
    then split over them as evenly as possible (the remainder to the first maps, ``split_worlds``) or given per map;
    ``spawn_override`` is None or one entry per map, ``cell`` applies to every map.  Map m owns a contiguous block of
    the worlds (``map_index`` gives the map of each, ``map_names`` their names), one launch steps all of them, and the
    observation, state and critic layouts are the single-map ones.  ``team_positions`` is bounded by the largest window.

    ``swappable_maps=True``: ``set_map(m, map)`` replaces map m of the live environment (a procedural layout, say:
    ``maps.generate_maze``) and resets its worlds, without re-creating the environment, its buffers or a captured
    rollout graph (``CatWorlds.set_map``).

    ``episode_statistics=True``: the step kernel tracks every world's return, as skrl's trainer does, within the same
    launch.  ``infos[agent]["episode"]`` is ``{"r": (N,) returns of that agent, "l": (N,) lengths}`` of the episodes that
    ended in the step (gymnasium's ``RecordEpisodeStatistics`` shape, valid where ``terminated``), and
    ``episode_statistics()`` sums up every episode since the last read, overall or per map.

    ``randomize``: domain randomisation of the dynamics, a spec for every map or a sequence of one spec (or None) per
    map, e.g. ``{"max_speed": {"thief": (125, 175)}, "termination_radius": (15, 25), "max_step_count": (300, 500)}``
    (a bare ``(lo, hi)`` applies to both teams; fields not named stay at the environment's values).  Every re-spawn
    draws a world's thrust and top speed per team, capture radius and time limit for its next episode, inside the step
    kernel.  ``world_params()``, ``set_world_params(...)`` and ``set_randomization(...)`` read and change them between
    steps (a curriculum); observation and state spaces do not change.

    ``scripted``: built-in controllers play chosen agents inside the step kernel, e.g. ``{"thief_0": "evade"}``
    (modes ``random``, ``chase``, ``evade``, ``none``; ``scripts.py``).  An empty dict turns them on with nobody
    scripted.  A controller decides from the agent's own observation that the last step or reset emitted, and the next
    step uses that decision instead of the caller's action.  ``set_scripted(spec, mask)`` changes the modes between steps
    (in place, graph-safe); ``step`` takes a mapping without the agents in ``scripted_agents``.
    """

    def __init__(self, map: Union[Map, Sequence[Map]], num_envs: Union[int, Sequence[int]], *, max_step_count: int = 400,
                 time_step: float = 1 / 60.0, device: Union[str, torch.device] = "cuda:0", seed: int = 0, gid0: int = 0,
                 physical_params: Optional[dict] = None, stale_shape_cache: bool = True,
                 spawn_override: Optional[Union[dict, Sequence[Optional[dict]]]] = None, cell: Optional[float] = None,
                 render_mode=None, final_observations: bool = False, swappable_maps: bool = False,
                 episode_statistics: bool = False,
                 randomize: Union[None, Mapping, Sequence[Optional[Mapping]]] = None,
                 scripted: Optional[Mapping[str, Union[str, int]]] = None):
        params = _make_params(max_step_count, time_step, physical_params, auto_reset=1, seed=int(seed),
                              stale_shape_cache=int(stale_shape_cache))
        self._params = params
        if isinstance(map, Map):
            self.maps = [map]
            self._cmap = compile_map(map, spawn_override=spawn_override, cell=cell)
            self._cmaps = [self._cmap]
            self._setup_common(map, self._cmap, params)
            self._w = CatWorlds(self._cmap, num_envs, device=device, gid0=gid0, params=params, want_f32=True, want_critic=True,
                                want_final=final_observations, swappable_maps=swappable_maps,
                                want_episode_stats=episode_statistics, param_ranges=randomize,
                                want_scripts=scripted is not None)
        else:
            self.maps = list(map)
            n = len(self.maps)
            counts = split_worlds(num_envs, n) if isinstance(num_envs, (int, np.integer)) else [int(c) for c in num_envs]
            if len(counts) != n:
                raise ValueError(f"{n} maps need {n} world counts, got {len(counts)}")
            overrides = [None] * n if spawn_override is None else list(spawn_override)
            if len(overrides) != n:
                raise ValueError(f"spawn_override: one entry per map ({n}), got {len(overrides)}")
            self._cmaps = [compile_map(m, spawn_override=o, cell=cell) for m, o in zip(self.maps, overrides)]
            self._cmap = self._cmaps[0]
            if any(c.agent_ids != self._cmap.agent_ids for c in self._cmaps):
                raise ValueError("every map of a mixed environment needs the same agents")
            window = (max(m.window_dimensions[0] for m in self.maps), max(m.window_dimensions[1] for m in self.maps))
            self._setup_common(self.maps[0], self._cmap, params, window=window)
            self._w = CatWorlds(self._cmaps, counts, device=device, gid0=gid0, params=params, want_f32=True,
                                want_critic=True, want_final=final_observations, swappable_maps=swappable_maps,
                                want_episode_stats=episode_statistics, param_ranges=randomize,
                                want_scripts=scripted is not None)
            num_envs = sum(counts)
        self._cell = cell
        self.map_names = [c.name for c in self._cmaps]
        self.map_index = self._w.map_index
        self.num_envs = int(num_envs)
        self.num_agents = len(self.possible_agents)
        self.agents = self.possible_agents[:]
        self.device = self._w.device
        self.render_mode = render_mode
        self.max_step_count = max_step_count
        self.state_spaces = {a: self.shared_observation_spaces for a in self.possible_agents}
        self.state_dim = self._w.S
        # the slot of a scripted agent a mapping leaves out of step(): the kernel never reads it
        self._script_zero = torch.zeros(self.num_envs, dtype=torch.int64, device=self.device)
        if scripted:
            self.set_scripted(scripted)

    @property
    def worlds(self) -> CatWorlds:
        return self._w

    def set_map(self, m: int, map: Map, spawn_override: Optional[dict] = None) -> torch.Tensor:
        """Replace map ``m`` of a ``swappable_maps`` environment by ``map`` (same agents; compiled with this
        environment's ``cell``) and reset its worlds; returns the (N,) bool mask of those worlds, whose observations in
        the step's output views are now their first ones on the new map.  Pass the mask to ``MAPPOLearner.note_reset``
        so that their recurrent states start afresh.  ``maps``, ``map_names`` and the shared observation spaces
        (``team_positions`` is bounded by the largest window) follow the new map."""
        cmap = compile_map(map, spawn_override=spawn_override, cell=self._cell)
        if cmap.agent_ids != self._cmap.agent_ids:
            raise ValueError("the new map needs the environment's agents")
        mask = self._w.set_map(m, cmap)
        self.maps[m] = map
        self._cmaps[m] = cmap
        self._cmap = self._cmaps[0]
        self.map_names[m] = cmap.name
        window = (max(mp.window_dimensions[0] for mp in self.maps), max(mp.window_dimensions[1] for mp in self.maps))
        self._setup_common(self.maps[0], self._cmap, self._params, window=window)
        _EnvCommon.get_nested_agent_observation_spaces.cache_clear()   # built from the old spaces
        self.state_spaces = {a: self.shared_observation_spaces for a in self.possible_agents}
        return mask

    def state_space_of(self, agent: str):
        return self.state_spaces[agent]

    def _obs_dict(self) -> Dict[str, torch.Tensor]:
        return self._views()[0]

    def _views(self):
        """The step's return values are fixed views of the kernel's output buffers, built once: per-agent
        observation / reward slices, and the u8 flags reinterpreted as bool (the kernel writes 0 / 1), so a step
        costs one kernel launch and no torch ops.  The same dict objects are returned by every call; their
        tensors are overwritten by the next step (copy what must outlive it, as skrl's memories do)."""
        v = getattr(self, "_cached_views", None)
        if v is None:
            w = self._w
            obs = {a: w.obs_f32[i] for i, a in enumerate(self.possible_agents)}
            rew = {a: w.reward[:, i:i + 1] for i, a in enumerate(self.possible_agents)}
            term = w.terminated.view(torch.bool).unsqueeze(1)
            trunc = w.truncated.view(torch.bool).unsqueeze(1)
            infos = {a: {"winner": w.winner} for a in self.possible_agents}
            if w.final_obs_f32 is not None:
                for i, a in enumerate(self.possible_agents):
                    infos[a]["final_observation"] = w.final_obs_f32[i]
            if w.episode_return is not None:
                for i, a in enumerate(self.possible_agents):
                    infos[a]["episode"] = {"r": w.episode_return[:, i], "l": w.episode_length}
            v = (obs, rew, {a: term for a in self.possible_agents}, {a: trunc for a in self.possible_agents}, infos)
            self._cached_views = v
        return v

    def reset(self, seed: Optional[int] = None, options: Optional[dict] = None):
        if seed is not None:
            self._w.set_seed(seed, restart_episodes=True)
        self._w.reset()
        return self._obs_dict(), {a: {} for a in self.possible_agents}

    def step(self, actions: Union[Mapping[str, torch.Tensor], torch.Tensor]):
        if isinstance(actions, Mapping):
            acts = [actions[a].reshape(-1) if a in actions or a not in self.scripted_agents else self._script_zero
                    for a in self.possible_agents]
            if all(t.dtype == torch.int64 and t.is_contiguous() and t.device == self.device for t in acts):
                self._w.step(acts)
            else:
                self._w.step(torch.stack([t.to(self.device) for t in acts], dim=1).to(torch.uint8).contiguous())
        else:
            self._w.step(actions)
        return self._views()

    def state(self) -> torch.Tensor:
        return self._w.state_f32

    def critic(self) -> torch.Tensor:
        """The critic's front end, written by the step kernel itself: the 4 ray channels ``LSTMValue`` cuts out of
        ``state()`` (``lstm_value_net.py:122-137``) as ``(N, 4, R)`` float32 — no slice / stack copies on the way."""
        return self._w.critic_f32

    def final_state(self) -> Optional[torch.Tensor]:
        """``state()`` of the last step of every episode that ended, (N, S) float32, valid where ``terminated``
        (None without ``final_observations``)."""
        return self._w.final_state_f32

    def final_critic(self) -> Optional[torch.Tensor]:
        """``critic()`` of the last step of every episode that ended, (N, 4, R) float32, valid where ``terminated``
        (None without ``final_observations``)."""
        return self._w.final_critic_f32

    def episode_statistics(self, reset: bool = False, by_map: bool = False, group=None) -> Dict:
        """What the episodes that ended since creation (or the last ``reset=True``) add up to, from the step kernel's
        per-map totals (one copy to the host): ``episodes``, ``captures``, ``timeouts``, ``capture_rate``, ``length``
        (mean / min / max) and per agent ``returns`` (mean / population std / min / max); None where no episode ended.
        ``by_map``: ``{"overall": ..., "maps": [one entry per map slot with "slot" and "map" (its name)]}``.  ``group``:
        a ``torch.distributed`` group whose ranks' totals are all-reduced first (collective: every rank calls it).
        ``reset`` zeroes this rank's totals after reading them.  Needs ``episode_statistics=True``."""
        from . import episodes
        raw = self._w.episode_totals_raw(reset)
        if group is not None:
            raw = episodes.allreduce_totals(raw, group)
        return episodes.summarize_maps(raw, self.possible_agents, self.map_names, by_map=by_map)

    def world_params(self) -> Dict[str, torch.Tensor]:
        """Every world's current dynamics, named device views (``CatWorlds.world_params``).  Needs ``randomize``."""
        return self._w.world_params()

    def set_world_params(self, mask: Optional[torch.Tensor] = None, **values) -> None:
        """Write worlds' dynamics directly (``CatWorlds.set_world_params``), e.g. ``termination_radius=15.0``."""
        self._w.set_world_params(mask, **values)

    def set_randomization(self, randomize: Union[None, Mapping, Sequence[Optional[Mapping]]]) -> None:
        """Replace the randomisation spec (one for every map, or one per map; ``None`` stops drawing, leaving the current
        values in place).  It applies from each world's next re-spawn.  Needs ``randomize`` at creation."""
        from . import world_params as wparams
        for slot, spec in enumerate(wparams.per_slot(randomize, len(self._cmaps))):
            self._w.set_param_ranges(slot, draw=spec is not None, **(spec or {}))

    def set_scripted(self, spec: Mapping[str, Union[str, int]], mask=None) -> None:
        """Set agents' modes, ``{"thief_0": "evade", "cop_0": "none"}``, in the worlds of the (N,) bool ``mask`` (all if
        None); agents not named keep theirs.  Checked before anything is written, then written in place (a captured
        graph stays valid).  Needs ``scripted`` at creation."""
        from . import scripts
        self._w.set_scripts(scripts.agent_modes(spec, self.possible_agents), mask)

    @property
    def scripted_agents(self) -> List[str]:
        """The agents scripted in every world (from the host mirror of the modes: no device sync)."""
        return [a for i, a in enumerate(self.possible_agents) if self._w.scripted_in(i) == "all"]

    def scripted_in(self, agent: str) -> str:
        """``"all"``, ``"none"`` or ``"some"``: in which worlds ``agent`` is scripted."""
        return self._w.scripted_in(self.possible_agents.index(agent))

    def render(self, world: int = 0):
        """``rgb_array`` of one world, drawn on that world's own map (numpy (W, H, 3) uint8 of that map's window):
        ``render.render_rgb`` bit for bit, drawn on the GPU."""
        cmap = self._cmaps[int(self._w.map_index[world])]
        frame = self._w.render_frames([int(world)])[0]
        return frame[:int(cmap.window[0]), :int(cmap.window[1])].cpu().numpy()

    def render_frames(self, worlds=None, rays: bool = False, downsample: int = 1, out: Optional[torch.Tensor] = None):
        """Frames of many worlds in one launch, on the device: ``CatWorlds.render_frames``."""
        return self._w.render_frames(worlds, rays=rays, downsample=downsample, out=out)

    def close(self) -> None:
        self._w.close()
