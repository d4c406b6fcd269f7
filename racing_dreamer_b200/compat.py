"""Gym-style dict API over the CUDA env step -- the drop-in for the reference's env path (SURVEY.md §8-b).

Two views of the same kernels:

* ``ReferenceEnv`` / ``make_reference_env``: the OUTERMOST interface of the reference's wrapper stack
  ``RaceCarBaseEnv -> RaceCarWrapper -> ActionRepeat -> ReduceActionSpace -> OccupancyMapObs -> FixedResetMode
  -> TimeLimit`` (+ the float32/int32 casts of ``Collect._convert``) [REF dreamer/dream.py:103-140;
  dreamer/wrappers.py:10-158,210-250,372-414], fused into ONE ``rd_step`` per agent step.
  ``dream.py::make_train_env/make_test_env`` can return this object instead of the wrapped PyBullet env.
* ``RaceCarGymCompat``: the ``racecar_gym.MultiAgentRaceEnv`` boundary itself (one 10 ms sim tick per ``step``,
  ``{'A': {'motor','steering'}}`` actions, ``reset(mode=...)``) [REF dreamer/wrappers.py:14-15,62-77,92], for
  callers that want to stack the reference's own unmodified wrapper classes on top.

Both are views of ONE world of a ``BatchedRaceEnv``: a single car ``'A'`` (the dreamer scenarios) or up to four cars
``'A'..'D'`` that see and hit each other (``n_agents`` / a multi-agent scenario YAML
[REF baselines/scenarios/max_progress/austria.yml:3-34; dreamer/dream.py:105-106]); results come from the same kernels
as the batched path.  Training-scale callers should use ``BatchedRaceEnv`` directly.
"""
from __future__ import annotations

import dataclasses
import types
from pathlib import Path
from typing import Dict as TDict, Optional, Union

import numpy as np
import torch

from . import _abi, spaces
from .env import BatchedRaceEnv, EnvConfig
from .maps import TrackMap, load_track

# task parameters of the reference's scenario files [REF dreamer/scenarios/max_progress/*.yml: laps 10;
# dreamer/scenarios/eval/*.yml: laps 1; both time_limit 180 s, terminate_on_collision, collision_reward -1]
SCENARIO_DEFAULTS = {
    "max_progress": dict(task="maximize_progress", laps=10, time_limit=180.0, terminate_on_collision=True,
                         collision_reward=-1.0),
    "eval": dict(task="maximize_progress", laps=1, time_limit=180.0, terminate_on_collision=True,
                 collision_reward=-1.0),
    "max_speed": dict(task="max_speed", laps=10, time_limit=180.0, terminate_on_collision=False,
                      collision_reward=-1.0),
}


AGENT_IDS = ("A", "B", "C", "D")


def baselines_config(tracks, n_envs: int, action_repeat: int = 4, mode: str = "train", **overrides) -> EnvConfig:
    """The model-free baselines' wrap chain (``BaselinesEnv``) as the config of a batched env of ``n_envs`` cars:
    flattened lidar normalised to [0, 1] (``normalize_obs='baselines'``), actions in [-1, 1] clipped by the env
    (``clip_actions``, no rescale), ``repeat_semantics='baselines'`` and the tick-based TimeLimit inside ActionRepeat
    [REF baselines/racing/experiments/acme/experiment.py:66-88; baselines/racing/experiments/sb3/sb_experiment.py:42-58].
    mode 'train': reset mode 'random', 2000 ticks; 'test': 'grid', 4000 ticks.  The max_progress scenario's task
    parameters unless ``overrides`` name others; ``overrides`` may set any ``EnvConfig`` field."""
    if mode not in ("train", "test"):
        raise ValueError("mode must be 'train' or 'test'")
    test = mode == "test"
    kw = dict(SCENARIO_DEFAULTS["max_progress"])
    kw.update(obs_type="lidar", action_repeat=int(action_repeat), reset_mode="grid" if test else "random",
              time_limit_steps=0, time_limit_ticks=4000 if test else 2000, rescale_actions=False, clip_actions=True,
              repeat_semantics="baselines", normalize_obs="baselines")
    kw.update(overrides)
    tracks = tuple(tracks) if isinstance(tracks, (list, tuple)) else (tracks,)
    return EnvConfig(tracks=tracks, n_envs=int(n_envs), **kw)


def load_scenario(path: Union[str, Path], agent_id: str = "A") -> dict:
    """Parse a reference scenario YAML [REF dreamer/scenarios/max_progress/austria.yml:1-10;
    baselines/scenarios/max_progress/austria.yml:1-34] into the keys ``EnvConfig`` understands:
    ``{'track': world.name, 'task': ..., 'laps': ..., ...}`` from agent ``agent_id``'s task, plus, for files with several
    agents, ``agents_per_world``, ``agent_tasks`` (one task name per agent, file order) and ``n_step_progress``."""
    import yaml
    spec = yaml.safe_load(Path(path).read_text())
    out = {"track": spec["world"]["name"]}
    agents = spec.get("agents", [])
    for agent in agents:
        task = agent.get("task", {})
        if task.get("task_name") == "n_step_progress" and "n_steps" in (task.get("params") or {}):
            out["n_step_progress"] = int(task["params"]["n_steps"])
        if agent.get("id") != agent_id:
            continue
        out["task"] = task.get("task_name", "maximize_progress")
        for k, v in (task.get("params") or {}).items():
            if k in ("laps", "time_limit", "terminate_on_collision", "collision_reward", "progress_reward",
                     "frame_reward"):
                out[k] = v
        out["sensors"] = list(agent.get("vehicle", {}).get("sensors", []))
    if len(agents) > 1:
        if len(agents) > _abi.MAX_AGENTS:
            raise ValueError(f"{path}: {len(agents)} agents, at most {_abi.MAX_AGENTS} cars per world are supported")
        out["agents_per_world"] = len(agents)
        out["agent_tasks"] = [a.get("task", {}).get("task_name", "maximize_progress") for a in agents]
        out["agent_ids"] = [str(a.get("id", AGENT_IDS[i])) for i, a in enumerate(agents)]
    return out


class _GridMap:
    """``scenario.world._maps[...]``: ``._map`` + ``.to_pixel(pose)`` [REF dreamer/wrappers.py:376,396-399]."""

    def __init__(self, tm: TrackMap, array: np.ndarray):
        self._tm = tm
        self._map = array

    @property
    def map(self):
        return self._map

    def to_pixel(self, pose):
        return self._tm.to_pixel(float(pose[0]), float(pose[1]))


def _scenario_of(tm: TrackMap):
    """Lazy stand-in for ``env.scenario`` [REF dreamer/wrappers.py:30-32; dreamer/evaluations/run_evaluation.py:48-49]."""
    class _Maps(dict):
        def __missing__(self, key):
            arr = {"occupancy": tm.full_drivable, "progress": tm.full_norm_distance_from_start,
                   "obstacle": tm.full_norm_distance_to_obstacle}[key]()
            self[key] = _GridMap(tm, arr)
            return self[key]
    world = types.SimpleNamespace(_maps=_Maps(), _config=types.SimpleNamespace(name=tm.name))
    return types.SimpleNamespace(world=world)


class _SingleAgentBase:
    """One world: a single car 'A' or n_agents cars 'A', 'B', ... (the name predates the multi-car worlds)."""
    agent_id = "A"
    _ids = ("A",)

    def _make(self, track, n_agents=1, agent_ids=None, order="manual", **cfg_kw):
        """track: one track or a list of tracks (racecar_gym's ChangingTrack* envs [REF dreamer/evaluations/make_env.py:
        6-11 order='manual'; baselines/racing/experiments/acme/experiment.py:90-93 order='sequential']): every map lives
        on the device, ``set_next_env()`` switches the world to the next one."""
        many = isinstance(track, (list, tuple))
        self._tms = [t if isinstance(t, TrackMap) else load_track(t) for t in (track if many else [track])]
        if order not in ("manual", "sequential"):
            raise ValueError("order must be 'manual' or 'sequential'")
        self._order = order
        self._track_idx = 0
        self._resets = 0
        self._tm = self._tms[0]
        n_agents = int(cfg_kw.get("agents_per_world", n_agents))
        cfg_kw["agents_per_world"] = n_agents
        self._ids = tuple(agent_ids) if agent_ids is not None else AGENT_IDS[:n_agents]
        if len(self._ids) != n_agents:
            raise ValueError("agent_ids must name every car of the world")
        self.agent_id = self._ids[0]
        self._env = BatchedRaceEnv(EnvConfig(tracks=tuple(self._tms), n_envs=n_agents, auto_reset=False,
                                             map_ids=[0] * n_agents, **cfg_kw), device=self._device)
        self._scenarios = [_scenario_of(tm) for tm in self._tms]
        self.scenario = self._scenarios[0]

    def set_next_env(self) -> None:
        """Switch to the next track of the list [REF dreamer/evaluations/run_evaluation.py:48-49]; takes effect with the
        next ``reset``, which the caller owes anyway."""
        self._track_idx = (self._track_idx + 1) % len(self._tms)
        self._tm = self._tms[self._track_idx]
        self.scenario = self._scenarios[self._track_idx]
        self._env.assign_maps([self._track_idx] * self.n_agents)
        self._needs_reset = True

    def _before_reset(self) -> None:
        # order='sequential': every reset but the first moves on to the next track
        if self._order == "sequential" and self._resets > 0 and len(self._tms) > 1:
            self.set_next_env()
        self._resets += 1

    @property
    def agent_ids(self):
        return list(self._ids)

    @property
    def n_agents(self):
        return len(self._ids)

    def _host(self) -> TDict[str, np.ndarray]:
        """One device->host read of every (tiny) result buffer of the world: arrays with leading dim n_agents."""
        buf = self._env.buf
        torch.cuda.current_stream(self._env.device).synchronize()
        return {k: v.cpu().numpy() for k, v in buf.items() if v is not None}

    def _info(self, h, f64=None, k: int = 0) -> dict:
        fl = int(h["flags"][k])
        pose = h["pose"][k].astype(np.float64)
        vel = h["velocity"][k].astype(np.float64)
        if f64 is not None:  # float64 pose straight from the state (racecar_gym reports float64)
            yaw = f64[_abi.S_YAW, k]
            pose = np.array([f64[_abi.S_X, k], f64[_abi.S_Y, k], 0.0, 0.0, 0.0, yaw - np.rint(yaw / (2 * np.pi)) * 2 * np.pi])
            v, b = f64[_abi.S_V, k], f64[_abi.S_SLIP, k]
            vel = np.array([v * np.cos(b), v * np.sin(b), 0.0, 0.0, 0.0, f64[_abi.S_YAWRATE, k]])
        opp = int(h["opponents"][k])
        return {"pose": pose, "velocity": vel, "progress": float(h["progress"][k]), "lap": int(h["lap"][k]),
                "time": float(h["time"][k]), "wrong_way": bool(fl & _abi.F_WRONG_WAY),
                "wall_collision": bool(fl & _abi.F_COLLISION),
                "opponent_collisions": [self._ids[j] for j in range(len(self._ids)) if (opp >> j) & 1],
                "rank": int(h["rank"][k]), "left_map": bool(fl & _abi.F_LEFT_MAP)}

    def render(self, mode: str = "birds_eye", agent: str = "A", **kwargs) -> np.ndarray:
        """RGB view (200, 200, 3) of the 10 m x 10 m around car ``agent``: 'birds_eye' = north up, 'follow' = the car's
        heading up; drivable area white, the cars of the world as filled body boxes (``agent`` red, the others blue).
        The reference renders these two views through PyBullet cameras [REF dreamer/wrappers.py:178-195; videos are
        written by callbacks.save_videos]; frames are not on the hot path, so this is a host-side map crop."""
        if mode not in ("birds_eye", "follow"):
            raise ValueError(f"render mode {mode!r}: expected 'birds_eye' or 'follow'")
        h = self._host()
        tm = self._tm
        k0 = self._ids.index(agent) if agent in self._ids else 0
        half, res = 100, tm.resolution
        x0, y0, yaw0 = float(h["pose"][k0][0]), float(h["pose"][k0][1]), float(h["pose"][k0][5])
        # world coordinates of every output pixel (row 0 = top)
        jj, ii = np.meshgrid(np.arange(2 * half) - half + 0.5, half - np.arange(2 * half) - 0.5)
        u, v = jj * res, ii * res
        if mode == "follow":   # heading up: image +v axis = car's x axis
            c, s = np.cos(yaw0), np.sin(yaw0)
            wx, wy = x0 + v * c + u * s, y0 + v * s - u * c
        else:
            wx, wy = x0 + u, y0 + v
        full = self.scenario.world._maps["occupancy"]._map
        col = np.floor((wx - tm.origin[0]) / res).astype(np.int64)
        row = full.shape[0] - 1 - np.floor((wy - tm.origin[1]) / res).astype(np.int64)
        ok = (row >= 0) & (row < full.shape[0]) & (col >= 0) & (col < full.shape[1])
        drv = np.zeros(wx.shape, bool)
        drv[ok] = full[row[ok], col[ok]]
        img = np.repeat((drv.astype(np.uint8) * 255)[..., None], 3, axis=2)
        hl, hw = 0.5 * float(self._env.cfg.vehicle.body_length), 0.5 * float(self._env.cfg.vehicle.body_width)
        for k in range(self.n_agents):
            px, py, pyaw = float(h["pose"][k][0]), float(h["pose"][k][1]), float(h["pose"][k][5])
            c, s = np.cos(pyaw), np.sin(pyaw)
            lx, ly = (wx - px) * c + (wy - py) * s, (wy - py) * c - (wx - px) * s
            img[(np.abs(lx) <= hl) & (np.abs(ly) <= hw)] = (255, 0, 0) if k == k0 else (0, 0, 255)
        return img

    def close(self):
        self._env.close()

    @property
    def launch_count(self) -> int:
        return self._env.launch_count


class ReferenceEnv(_SingleAgentBase):
    """Fused equivalent of the reference's fully wrapped env (see module docstring).

    ``reset() -> {'A': obs}``; ``step({'A': a}) -> (obs, rewards, dones, infos)`` with ``a`` a length-2 array
    ``[motor, steering]`` in [-1, 1] [REF dreamer/wrappers.py:55-63,129-134].  obs keys: ``lidar`` f32[1080],
    ``pose`` f32[6], ``velocity`` f32[6], ``speed`` f32 scalar, ``lidar_occupancy`` u8[64,64,1] (zeros on reset
    [REF dreamer/wrappers.py:410-414]) -- dtypes as ``Collect._convert`` leaves them at precision 32.
    """

    def __init__(self, track="austria", task="max_progress", action_repeat=4, time_limit_steps=None,
                 reset_mode=None, occupancy=True, device=None, scenario: Optional[str] = None, n_agents: int = 1,
                 order: str = "manual", **overrides):
        """n_agents > 1 (or a scenario file with several agents): one world of cars 'A', 'B', ...; every dict below then
        has one entry per car, ActionRepeat stops when ANY car is done, TimeLimit sets every done
        [REF dreamer/wrappers.py:107-116,147-154]; reset_mode defaults to 'random_ball' for several cars and 'random'
        for one [REF dreamer/dream.py:105-108]."""
        self._device = device
        params = dict(SCENARIO_DEFAULTS.get(task, SCENARIO_DEFAULTS["max_progress"]))
        ids = None
        if scenario is not None:
            sc = load_scenario(scenario)
            track = sc.pop("track", track)
            sc.pop("sensors", None)
            ids = sc.pop("agent_ids", None)
            params.update(sc)
        params.update(overrides)
        n_agents = int(params.pop("agents_per_world", n_agents))
        if reset_mode is None:
            reset_mode = "random_ball" if n_agents > 1 else "random"
        if time_limit_steps is None:  # dream.py: time_limit_train 2000 sim ticks / action_repeat [REF dreamer/dream.py:57,109]
            time_limit_steps = -(-2000 // int(action_repeat))   # TimeLimit(2000 / action_repeat) tests `step >= duration`: ceil
        self._make(track, n_agents=n_agents, agent_ids=ids, order=order, action_repeat=int(action_repeat), reset_mode=reset_mode,
                   obs_type="lidar_occupancy" if occupancy else "lidar", time_limit_steps=int(time_limit_steps),
                   rescale_actions=True, **params)
        self._occupancy = occupancy
        self._needs_reset = True
        self._action = torch.zeros((self.n_agents, 2), dtype=torch.float32, device=self._env.device)

    @property
    def observation_space(self):
        box = spaces.Box
        sp = {"lidar": box(0.0, 15.0, shape=(1080,), dtype=np.float32),
              "pose": box(-100.0, 100.0, shape=(6,), dtype=np.float32),
              "velocity": box(-10.0, 10.0, shape=(6,), dtype=np.float32),
              "speed": box(-np.inf, np.inf, shape=(1,), dtype=np.float32)}  # [REF dreamer/wrappers.py:50]
        if self._occupancy:
            sp["lidar_occupancy"] = box(0, 1, shape=(64, 64, 1), dtype=np.uint8)  # [REF dreamer/wrappers.py:380-385]
        return spaces.Dict({aid: spaces.Dict(dict(sp)) for aid in self._ids})

    @property
    def action_space(self):  # [REF dreamer/wrappers.py:55-60]: Box(append(motor.low, steering.low), ...)
        return spaces.Dict({aid: spaces.Box(np.array([-1.0, -1.0], np.float32), np.array([1.0, 1.0], np.float32))
                            for aid in self._ids})

    def _obs(self, h, reset: bool):
        out = {}
        for k, aid in enumerate(self._ids):
            obs = {"lidar": h["lidar"][k], "pose": h["pose"][k], "velocity": h["velocity"][k],
                   "speed": np.float32(0.0) if reset else np.float32(h["speed"][k])}
            if self._occupancy:
                obs["lidar_occupancy"] = h["occupancy"][k]
            out[aid] = obs
        return out

    def reset(self, mode: Optional[str] = None):
        self._before_reset()
        self._env.reset(mode=mode)
        self._needs_reset = False
        return self._obs(self._host(), reset=True)

    def step(self, actions):
        assert not self._needs_reset, "Must reset environment."  # [REF dreamer/wrappers.py:148]
        a = np.stack([np.asarray(actions[aid], dtype=np.float32).reshape(2) for aid in self._ids])
        self._action.copy_(torch.from_numpy(a))
        self._env.step(self._action)
        h = self._host()
        dones = {aid: bool(h["done"][k]) for k, aid in enumerate(self._ids)}
        self._needs_reset = any(dones.values())   # the world is over for everybody [REF dreamer/tools.py:178-179]
        return (self._obs(h, reset=False), {aid: float(h["reward"][k]) for k, aid in enumerate(self._ids)}, dones,
                {aid: self._info(h, k=k) for k, aid in enumerate(self._ids)})


class RaceCarGymCompat(_SingleAgentBase):
    """``racecar_gym.envs.MultiAgentRaceEnv``-shaped view: one sim tick per ``step`` (see module docstring)."""

    def __init__(self, track="austria", task="max_progress", device=None, scenario: Optional[str] = None,
                 n_agents: int = 1, order: str = "manual", **overrides):
        self._device = device
        params = dict(SCENARIO_DEFAULTS.get(task, SCENARIO_DEFAULTS["max_progress"]))
        ids = None
        if scenario is not None:
            sc = load_scenario(scenario)
            track = sc.pop("track", track)
            sc.pop("sensors", None)
            ids = sc.pop("agent_ids", None)
            params.update(sc)
        params.update(overrides)
        n_agents = int(params.pop("agents_per_world", n_agents))
        self._make(track, n_agents=n_agents, agent_ids=ids, order=order, action_repeat=1, rescale_actions=False, obs_type="lidar",
                   time_limit_steps=0, **params)
        self._action = torch.zeros((self.n_agents, 2), dtype=torch.float32, device=self._env.device)

    @property
    def observation_space(self):
        box = spaces.Box
        return spaces.Dict({aid: spaces.Dict({
            "lidar": box(0.0, 15.0, shape=(1080,), dtype=np.float64),
            "pose": box(-100.0, 100.0, shape=(6,), dtype=np.float64),
            "velocity": box(-10.0, 10.0, shape=(6,), dtype=np.float64)}) for aid in self._ids})

    @property
    def action_space(self):
        box = spaces.Box
        return spaces.Dict({aid: spaces.Dict({
            "motor": box(-1.0, 1.0, shape=(1,), dtype=np.float64),
            "steering": box(-1.0, 1.0, shape=(1,), dtype=np.float64)}) for aid in self._ids})

    def _state(self):
        f, _ = self._env.get_state()
        return f.cpu().numpy()

    def _obs(self, h, infos):
        return {aid: {"lidar": h["lidar"][k].astype(np.float64), "pose": infos[aid]["pose"],
                      "velocity": infos[aid]["velocity"]} for k, aid in enumerate(self._ids)}

    def _infos(self, h):
        f64 = self._state()
        return {aid: self._info(h, f64, k) for k, aid in enumerate(self._ids)}

    def reset(self, mode: str = "grid"):
        self._before_reset()
        self._env.reset(mode=mode)
        h = self._host()
        return self._obs(h, self._infos(h))

    def step(self, actions):
        cmd = np.array([[float(np.asarray(actions[aid]["motor"]).reshape(-1)[0]),
                         float(np.asarray(actions[aid]["steering"]).reshape(-1)[0])] for aid in self._ids], dtype=np.float32)
        # racecar_gym keeps stepping after a terminal tick; the wrappers above decide when to reset
        _, i = self._env.get_state()
        i[_abi.I_FLAGS] &= ~_abi.F_NEEDS_RESET
        self._env.set_state(None, i)
        self._action.copy_(torch.from_numpy(cmd))
        self._env.step(self._action)
        h = self._host()
        infos = self._infos(h)
        return (self._obs(h, infos), {aid: float(h["reward"][k]) for k, aid in enumerate(self._ids)},
                {aid: bool(h["done"][k]) for k, aid in enumerate(self._ids)}, infos)


class SingleAgentRaceCompat:
    """``racecar_gym.envs.SingleAgentRaceEnv`` / ``ChangingTrackSingleAgentRaceEnv``-shaped view -- what the model-free
    baselines build their wrapper chain on [REF baselines/racing/experiments/acme/experiment.py:66-93;
    baselines/racing/experiments/sb3/sb_experiment.py:60-64]: one car, one sim tick per ``step``, observations / rewards /
    dones NOT keyed by agent id, ``reset(mode=...)``; a list of tracks + ``order='sequential'`` moves to the next track at
    every reset.  The reference's own ``FilterObservation -> Flatten -> NormalizeObservations -> FixedResetMode ->
    TimeLimit -> ActionRepeat`` stack goes on top unchanged (``EnvConfig(clip_actions=True, rescale_actions=False,
    repeat_semantics='baselines')`` is its fused form)."""

    def __init__(self, track="austria", task="max_progress", device=None, scenario: Optional[str] = None,
                 order: str = "sequential", **overrides):
        self._env = RaceCarGymCompat(track, task, device=device, scenario=scenario, n_agents=1, order=order, **overrides)
        self._id = self._env.agent_id

    @property
    def scenario(self):
        return self._env.scenario

    @property
    def observation_space(self):
        return self._env.observation_space[self._id]

    @property
    def action_space(self):
        return self._env.action_space[self._id]

    def reset(self, mode: str = "grid"):
        return self._env.reset(mode=mode)[self._id]

    def step(self, action):
        obs, rew, done, info = self._env.step({self._id: action})
        return obs[self._id], rew[self._id], done[self._id], info[self._id]

    def set_next_env(self) -> None:
        self._env.set_next_env()

    def render(self, mode: str = "follow", **kwargs):
        return self._env.render(mode=mode, agent=self._id)

    def close(self):
        self._env.close()


class BaselinesEnv(_SingleAgentBase):
    """Fused equivalent of the model-free agents' wrap chains [REF baselines/racing/experiments/acme/experiment.py:66-88
    _wrap_training / _wrap_test; baselines/racing/experiments/sb3/sb_experiment.py:42-58]:

        ChangingTrackSingleAgentRaceEnv -> FilterObservation(['lidar']) -> Flatten -> NormalizeObservations
        (-> InfoToObservation) -> FixedResetMode -> TimeLimit(max_episode_steps, in sim ticks) -> ActionRepeat(n)
        (-> SinglePrecisionWrapper)

    as ONE ``rd_step`` per agent step: the action clip of ``Flatten``, ``(x - low) / (high - low)`` of
    ``NormalizeObservations`` [REF baselines/racing/environment/single_agent.py:55-56,66-99] and the tick-based time limit
    run inside the kernels (``clip_actions``, ``normalize_obs='baselines'``, ``time_limit_ticks``,
    ``repeat_semantics='baselines'``).

    ``mode='train'``: ``reset() -> float32[1080]`` (the flattened, normalised scan), reset mode 'random', 2000 ticks.
    ``mode='test'``:  ``reset() -> {'lidar': float32[1080]}``; after a step the dict also carries ``info_<key>`` for every
    info key, as ``InfoToObservation`` adds them [REF baselines/racing/environment/common.py:31-39]; reset mode 'grid',
    4000 ticks.  ``step(action[2]) -> (obs, reward, done, info)`` -- not keyed by agent id (``SingleAgentRaceEnv``);
    ``info['TimeLimit.truncated']`` is set the way gym's TimeLimit does.  A list of tracks + ``order='sequential'`` moves
    to the next track at every reset [REF acme/experiment.py:90-93]."""

    def __init__(self, track="austria", task="max_progress", action_repeat: int = 4, mode: str = "train",
                 time_limit: Optional[int] = None, device=None, scenario: Optional[str] = None,
                 order: str = "sequential", **overrides):
        if mode not in ("train", "test"):
            raise ValueError("mode must be 'train' or 'test'")
        self._device = device
        self._test = mode == "test"
        params = dict(SCENARIO_DEFAULTS.get(task, SCENARIO_DEFAULTS["max_progress"]))
        if scenario is not None:
            sc = load_scenario(scenario)
            track = sc.pop("track", track)
            for k in ("sensors", "agent_ids", "agents_per_world", "agent_tasks"):   # SingleAgentScenario: agent A only
                sc.pop(k, None)
            params.update(sc)
        params.update(overrides)
        if time_limit is not None:
            params["time_limit_ticks"] = int(time_limit)
        ec = baselines_config(track, 1, action_repeat, mode, **params)
        self._limit = int(ec.time_limit_ticks)
        self._reset_mode = ec.reset_mode
        # _make sets the tracks, the car count and the manual resets itself
        self._make(track, n_agents=1, order=order, **{f.name: getattr(ec, f.name) for f in dataclasses.fields(ec)
                                                      if f.name not in ("tracks", "n_envs", "map_ids", "auto_reset")})
        self._needs_reset = True
        self._action = torch.zeros((1, 2), dtype=torch.float32, device=self._env.device)

    @property
    def observation_space(self):
        lidar = spaces.Box(0.0, 1.0, shape=(1080,), dtype=np.float32)   # NormalizeObservations: zeros .. ones
        return spaces.Dict({"lidar": lidar}) if self._test else lidar

    @property
    def action_space(self):  # Flatten: Box(-1, 1, shape (2,)) = [motor, steering] [REF single_agent.py:49-52]
        return spaces.Box(np.array([-1.0, -1.0], np.float32), np.array([1.0, 1.0], np.float32))

    def _obs(self, h, info=None):
        lidar = h["lidar"][0]
        if not self._test:
            return lidar
        obs = {"lidar": lidar}
        for k, v in (info or {}).items():   # InfoToObservation sits inside TimeLimit: it never sees 'TimeLimit.truncated'
            if k != "TimeLimit.truncated":
                obs[f"info_{k}"] = v
        return obs

    def reset(self, mode: Optional[str] = None):
        self._before_reset()
        self._env.reset(mode=mode or self._reset_mode)
        self._needs_reset = False
        return self._obs(self._host())

    def step(self, action):
        assert not self._needs_reset, "Cannot call env.step() before calling reset()"   # gym TimeLimit's assertion
        self._action.copy_(torch.from_numpy(np.asarray(action, dtype=np.float32).reshape(1, 2)))
        self._env.step(self._action)
        h = self._host()
        done = bool(h["done"][0])
        info = self._info(h)
        # gym TimeLimit: the step that reaches max_episode_steps reports whether the env itself was done
        ticks = int(round(float(h["time"][0]) / float(self._env.cfg.dt)))
        if done and ticks >= self._limit:
            task_done = bool(info["wall_collision"] and int(self._env.cfg.terminate_on_collision)) or \
                info["lap"] > int(self._env.cfg.laps) or info["time"] > float(self._env.cfg.time_limit)
            info["TimeLimit.truncated"] = not task_done
        self._needs_reset = done
        return self._obs(h, info), float(h["reward"][0]), done, info


def make_reference_env(track: str, task: str = "max_progress", action_repeat: int = 4, mode: str = "train",
                       device=None, **kw) -> ReferenceEnv:
    """``make_train_env`` / ``make_test_env`` of dream.py without the PyBullet sim [REF dreamer/dream.py:103-131]:
    train = reset mode 'random', TimeLimit 2000/action_repeat; test = 'grid', 4000/action_repeat.  dream.py passes the
    float quotient and TimeLimit ends the episode at `step >= duration` [REF dreamer/wrappers.py:150], i.e. after
    ceil(limit / action_repeat) agent steps."""
    if mode == "train":  # 'random' for one car, 'random_ball' for several [REF dreamer/dream.py:105-108]
        return ReferenceEnv(track, task, action_repeat, time_limit_steps=-(-2000 // action_repeat), reset_mode=None,
                            device=device, **kw)
    return ReferenceEnv(track, task, action_repeat, time_limit_steps=-(-4000 // action_repeat), reset_mode="grid",
                        device=device, **kw)
