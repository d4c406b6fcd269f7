"""Episode store -- the wire format between the env and Dreamer's replay (SURVEY.md §8-f row 1).

Restates, for a BATCH of envs, what the reference does per env:

* ``Collect.step/reset`` [REF dreamer/wrappers.py:198-250]: every transition is the observation dict plus ``action``,
  ``reward``, ``discount = 1 - done``, ``progress = lap + progress - 1`` and ``time``; the first row of an episode is the
  reset observation with zero action, reward 0, discount 1, progress -1, time 0; floats are cast to float32, signed
  ints to int32, uint8 stays (precision 32).
* ``callbacks.save_episodes`` [REF dreamer/callbacks.py:41-53]: one ``{timestamp}-{uuid}-{length}.npz`` per episode,
  ``np.savez_compressed`` of the stacked rows.
* ``tools.count_episodes / load_episodes`` [REF dreamer/tools.py:224-264]: episode counting from file names and the
  random fixed-length chunk sampler that feeds the learner.

``EpisodeRecorder`` drives any env with the host-facing interface (``reset(mask=None, mode=None) -> dict`` and
``step(actions) -> dict`` of numpy arrays keyed lidar, pose, velocity, speed, reward, done, progress, lap, time
[, occupancy]) -- ``HostSteppedEnv`` on the GPU.  The env must be created with ``auto_reset=False``: the terminal
observation belongs to the finished episode (as in the reference), and the recorder resets exactly the finished envs.
"""
from __future__ import annotations

import datetime
import io
import pathlib
import uuid
from typing import Callable, Dict, Iterator, List, Optional, Sequence

import numpy as np

OBS_KEYS = ("lidar", "pose", "velocity", "speed", "lidar_occupancy")     # order of the reference's obs dict
EXTRA_KEYS = ("action", "reward", "discount", "progress", "time")


def save_episodes(directory, episodes: Sequence[Dict[str, np.ndarray]]) -> List[pathlib.Path]:
    """[REF dreamer/callbacks.py:41-53] -- same file naming and container; returns the paths written."""
    directory = pathlib.Path(directory).expanduser()
    directory.mkdir(parents=True, exist_ok=True)
    timestamp = datetime.datetime.now().strftime("%Y%m%dT%H%M%S")
    out = []
    for episode in episodes:
        identifier = str(uuid.uuid4().hex)
        length = len(episode["reward"])
        filename = directory / f"{timestamp}-{identifier}-{length}.npz"
        with io.BytesIO() as f1:
            np.savez_compressed(f1, **episode)
            f1.seek(0)
            with filename.open("wb") as f2:
                f2.write(f1.read())
        out.append(filename)
    return out


def count_episodes(directory):
    """(episodes, agent steps) from the file names [REF dreamer/tools.py:224-228]."""
    filenames = pathlib.Path(directory).expanduser().glob("*.npz")
    lengths = [int(n.stem.rsplit("-", 1)[-1]) - 1 for n in filenames]
    return len(lengths), sum(lengths)


def load_episodes(directory, rescan, length=None, balance=False, seed=0) -> Iterator[Dict[str, np.ndarray]]:
    """Endless sampler of (chunks of) stored episodes with the reference's RandomState call sequence
    [REF dreamer/tools.py:235-264].  Files are visited in sorted order so that the stream is reproducible."""
    directory = pathlib.Path(directory).expanduser()
    random = np.random.RandomState(seed)
    cache = {}
    while True:
        for filename in sorted(directory.glob("*.npz")):
            if filename not in cache:
                try:
                    with filename.open("rb") as f:
                        episode = np.load(f)
                        episode = {k: episode[k] for k in episode.keys()}
                except Exception as e:  # noqa: BLE001 - a half-written file must not stop training (reference behaviour)
                    print(f"Could not load episode: {e}")
                    continue
                cache[filename] = episode
        keys = list(cache.keys())
        for index in random.choice(len(keys), rescan):
            episode = cache[keys[index]]
            if length:
                total = len(next(iter(episode.values())))
                available = total - length
                if available < 1:
                    print(f"[Info] Skipped short episode of length {available}.")
                    continue
                if balance:
                    index = min(random.randint(0, total), available)
                else:
                    index = int(random.randint(0, available + 1))
                episode = {k: v[index: index + length] for k, v in episode.items()}
            yield episode


def _convert(value: np.ndarray, precision: int = 32) -> np.ndarray:
    """[REF dreamer/wrappers.py:240-250]"""
    value = np.asarray(value)
    if np.issubdtype(value.dtype, np.floating):
        dtype = {16: np.float16, 32: np.float32, 64: np.float64}[precision]
    elif np.issubdtype(value.dtype, np.signedinteger):
        dtype = {16: np.int16, 32: np.int32, 64: np.int64}[precision]
    elif np.issubdtype(value.dtype, np.uint8):
        dtype = np.uint8
    else:
        raise NotImplementedError(value.dtype)
    return value.astype(dtype)


class EpisodeRecorder:
    """Batched ``Collect``: records every env's transitions and hands finished episodes to the callbacks.

    ``callbacks``: callables taking a list with ONE episode dict (the reference calls its callbacks with one episode per
    agent of a single env [REF dreamer/wrappers.py:221-225]; here every finished env yields its own call).
    Storage is a preallocated ``[max_len + 1, n_envs, ...]`` array per key, filled column-wise; ``max_len`` must cover the
    env's TimeLimit.
    """

    def __init__(self, env, max_len: int, callbacks: Sequence[Callable] = (), precision: int = 32,
                 reset_mode: Optional[str] = None, keep_obs: Sequence[str] = OBS_KEYS,
                 agents_per_world: Optional[int] = None):
        """agents_per_world (default: the env's own ``cfg.agents_per_world``): for worlds of several cars the episodes of
        ALL cars of a world end at the step in which any of them is done -- the reference resets the world then
        [REF dreamer/tools.py:178-179] -- and the callbacks get one list with the world's episodes, agent A first, exactly
        what the reference's Collect passes for its single world [REF dreamer/wrappers.py:221-225]."""
        self.env = env
        self.n = int(env.n)
        cfg = getattr(env, "cfg", None) or getattr(getattr(env, "env", None), "cfg", None)
        A = agents_per_world if agents_per_world is not None else int(getattr(cfg, "agents_per_world", 1) or 1)
        self.agents = max(1, int(A))
        # Collect stores the TERMINAL observation of an episode and resets afterwards [REF dreamer/wrappers.py:210-226]; an
        # auto-resetting env has already replaced it with the first observation of the next episode (and advanced the
        # reset counters) by the time the recorder sees the done flag.
        if cfg is not None and int(getattr(cfg, "auto_reset", 0)):
            raise ValueError("EpisodeRecorder needs an env created with auto_reset=False: it resets finished envs itself, "
                             "after storing their terminal observation")
        if self.n % self.agents:
            raise ValueError("n_envs must be a multiple of agents_per_world")
        self.max_len = int(max_len)
        self.callbacks = tuple(callbacks)
        self.precision = precision
        self.reset_mode = reset_mode
        self.keep_obs = tuple(keep_obs)
        self._store: Dict[str, np.ndarray] = {}
        self._len = np.zeros(self.n, np.int64)
        self.episodes_done = 0

    # -- storage --
    def _obs_of(self, out: Dict[str, np.ndarray], reset: bool) -> Dict[str, np.ndarray]:
        obs = {"lidar": out["lidar"], "pose": out["pose"], "velocity": out["velocity"],
               "speed": np.zeros_like(out["speed"]) if reset else out["speed"]}       # [REF dreamer/wrappers.py:66,74]
        if "occupancy" in out:
            obs["lidar_occupancy"] = out["occupancy"]
        return {k: v for k, v in obs.items() if k in self.keep_obs}

    def _put(self, rows: Dict[str, np.ndarray], envs: np.ndarray) -> None:
        """Append one row per env in `envs` (values are [len(envs), ...])."""
        t = self._len[envs]
        if np.any(t > self.max_len):
            raise RuntimeError("episode longer than max_len: size the recorder to the env's TimeLimit")
        for k, v in rows.items():
            v = _convert(v, self.precision)
            if k not in self._store:
                self._store[k] = np.zeros((self.max_len + 1, self.n) + v.shape[1:], v.dtype)
            self._store[k][t, envs] = v
        self._len[envs] = t + 1

    def _flush(self, envs: np.ndarray) -> None:
        A = self.agents
        for e in envs[::A] if A > 1 else envs:      # worlds: `envs` holds whole worlds, one callback per world
            group = range(e, e + A) if A > 1 else (e,)
            episodes = []
            for c in group:
                n = int(self._len[c])
                episodes.append({k: self._store[k][:n, c].copy() for k in self._store})
                self._len[c] = 0
            self.episodes_done += len(episodes)
            for cb in self.callbacks:
                cb(episodes)

    # -- env API --
    def reset(self, mask: Optional[np.ndarray] = None) -> Dict[str, np.ndarray]:
        out = self.env.reset(mask=mask, mode=self.reset_mode)
        envs = np.arange(self.n) if mask is None else np.flatnonzero(np.asarray(mask))
        self._len[envs] = 0
        m = len(envs)
        rows = {k: v[envs] for k, v in self._obs_of(out, reset=True).items()}
        rows.update(action=np.zeros((m, 2), np.float32), reward=np.zeros(m, np.float32), discount=np.ones(m, np.float32),
                    progress=-np.ones(m, np.float32), time=np.zeros(m, np.float32))   # [REF dreamer/wrappers.py:228-238]
        self._put(rows, envs)
        return out

    def step(self, actions: np.ndarray, auto_reset: bool = True) -> Dict[str, np.ndarray]:
        """One env step for the whole batch; finished envs are flushed to the callbacks and (auto_reset) reset, so the
        dict returned holds, for those envs, the first observation of their next episode -- `done`/`reward` stay the
        finished step's."""
        actions = np.asarray(actions, np.float32)
        out = self.env.step(actions)
        live = np.flatnonzero(self._len > 0)           # envs inside an episode (frozen ones were flushed already)
        done = out["done"].astype(bool)
        rows = {k: v[live] for k, v in self._obs_of(out, reset=False).items()}
        rows.update(action=actions[live], reward=out["reward"][live],
                    discount=(1.0 - done[live].astype(np.float64)),
                    progress=out["lap"][live].astype(np.float64) + out["progress"][live].astype(np.float64) - 1.0,
                    time=out["time"][live])                                           # [REF dreamer/wrappers.py:214-219]
        self._put(rows, live)
        if self.agents > 1:     # a world is over for all of its cars as soon as one is done
            done = np.repeat(done.reshape(-1, self.agents).any(axis=1), self.agents)
        finished = live[done[live]]
        if finished.size:
            reward, done_flags = out["reward"].copy(), out["done"].copy()
            self._flush(finished)
            if auto_reset:
                mask = np.zeros(self.n, np.uint8)
                mask[finished] = 1
                out = dict(self.reset(mask))
                out["reward"], out["done"] = reward, done_flags
        return out


def max_episode_steps(cfg) -> Optional[int]:
    """Longest episode an ``rd_config`` allows, in agent steps (None: unbounded) -- what sizes a ``DeviceEpisodeStore``:
    ``time_limit_steps``, ``time_limit_ticks / action_repeat`` (rounded up) and, for tasks that end at
    ``time > time_limit``, that tick (at most ``floor(time_limit / dt) + 2`` ticks after the reset, allowing for the
    rounding of the time accumulated tick by tick) in agent steps.  A world of cars ends with its first car."""
    R = int(cfg.action_repeat)
    bounds = []
    if int(cfg.time_limit_steps) > 0:
        bounds.append(int(cfg.time_limit_steps))
    if int(cfg.time_limit_ticks) > 0:
        bounds.append(-(-int(cfg.time_limit_ticks) // R))
    A = int(cfg.agents_per_world)
    tasks = [int(cfg.agent_task[a]) for a in range(A)] if A > 1 else [int(cfg.task)]
    from . import _abi
    timed = any(t != _abi.TASK_MAX_SPEED for t in tasks)   # max_speed has no time limit of its own
    tl, dt = float(cfg.time_limit), float(cfg.dt)
    if timed and tl >= 0.0 and tl / dt < 1e15:
        bounds.append(int(np.ceil((np.floor(tl / dt) + 2.0) / R)))
    return min(bounds) if bounds else None


# keys of the dict DeviceEpisodeStore.step / reset return: those of HostSteppedEnv (what EpisodeRecorder.step returns)
_ENV_OUT_KEYS = ("lidar", "occupancy", "pose", "velocity", "speed", "reward", "done", "progress", "lap", "time", "flags",
                 "rank", "opponents", "wrong_way", "wall_collision")


class DeviceEpisodeStore:
    """``EpisodeRecorder`` on the device: records the ``Collect`` rows of every env of a ``BatchedRaceEnv`` into rings in
    GPU memory (include/rd_env.h ``rd_store_*``, kernels in csrc/rd_store.cuh) and samples ``load_episodes``-style
    fixed-length chunks as CUDA tensors ``[B, L, ...]``.

    The committed episodes are, bit for bit, those ``EpisodeRecorder`` over ``HostSteppedEnv`` hands to its callbacks for
    the same config, seed and actions, in the same order (``episodes()``).  Each env keeps a ring of ``capacity_rows``
    rows (memory: n_envs x capacity_rows x row bytes); an env's oldest episodes are evicted as its ring wraps.
    ``capacity_rows`` must exceed ``max_episode_steps(env.cfg)``.  ``seed`` keys the sampler's Philox stream."""

    def __init__(self, env, capacity_rows: int, precision: int = 32, keep_obs: Sequence[str] = OBS_KEYS,
                 reset_mode: Optional[str] = None, seed: int = 0):
        import ctypes as C
        from . import _abi
        self._C, self._abi = C, _abi
        self.env = env
        cfg = env.cfg
        if int(cfg.auto_reset):
            raise ValueError("DeviceEpisodeStore needs an env created with auto_reset=False: it resets finished envs "
                             "itself, after storing their terminal observation")
        occ = bool(cfg.obs_flags & _abi.OBS_OCCUPANCY)
        self.obs_keys = tuple(k for k in OBS_KEYS if k in keep_obs and (k != "lidar_occupancy" or occ))
        self.keys = self.obs_keys + EXTRA_KEYS
        self.precision = int(precision)
        self.capacity_rows = int(capacity_rows)
        sc = _abi.RdStoreConfig()
        sc.capacity_rows = self.capacity_rows
        sc.precision = self.precision
        sc.keep_obs = sum(_abi.STORE_KEYS[k] for k in self.obs_keys)
        sc.reset_mode = -1 if reset_mode is None else _abi.RESET_MODES[reset_mode]
        sc.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self._sc = sc
        import torch
        self._torch = torch
        fdt = torch.float16 if self.precision == 16 else torch.float32
        self._spec = {"lidar": ((env.n_beams,), fdt), "pose": ((6,), fdt), "velocity": ((6,), fdt), "speed": ((), fdt),
                      "lidar_occupancy": ((64, 64, 1), torch.uint8), "action": ((2,), fdt), "reward": ((), fdt),
                      "discount": ((), fdt), "progress": ((), fdt), "time": ((), fdt)}
        with torch.cuda.device(env.device):
            env._check(env.lib.rd_store_init(env._handle, C.byref(sc)))

    # -- recording --
    def _outputs(self):
        return {k: self.env.buf[k] for k in _ENV_OUT_KEYS if self.env.buf.get(k) is not None}

    def reset(self):
        """Resets every env and starts its first episode (episodes in progress are dropped, held ones kept).  Returns the
        env's output tensors, keyed like ``HostSteppedEnv.reset``."""
        env = self.env
        with self._torch.cuda.device(env.device):
            env._check(env.lib.rd_store_reset(env._handle, self._C.byref(env._out), env._stream()))
        return self._outputs()

    def step(self, actions):
        """One env step for the whole batch, recorded; finished envs are committed and reset, so the dict returned (device
        tensors keyed like ``HostSteppedEnv.step``) holds, for those envs, the first observation of their next episode --
        ``reward`` / ``done`` stay the finished step's (``EpisodeRecorder.step``)."""
        env = self.env
        a = actions if isinstance(actions, self._torch.Tensor) else self._torch.from_numpy(np.asarray(actions, np.float32))
        if tuple(a.shape) != (env.n, 2):
            raise ValueError(f"actions must have shape ({env.n}, 2), got {tuple(a.shape)}")
        if a.dtype != self._torch.float32 or a.device != env.device or not a.is_contiguous():
            env._actions.copy_(a, non_blocking=True)
            a = env._actions
        with self._torch.cuda.device(env.device):
            env._check(env.lib.rd_store_step(env._handle, a.data_ptr(), self._C.byref(env._out), env._stream()))
        return self._outputs()

    # -- sampling --
    def sample(self, batch: Optional[int] = None, length: Optional[int] = None, balance: bool = False,
               indices=None, check: bool = False) -> Dict[str, "torch.Tensor"]:
        """``batch`` chunks of ``length`` rows as CUDA tensors ``[B, L, ...]`` per key, plus ``episode_id`` i64 [B] and
        ``start`` i32 [B].  Drawn uniformly over the held episodes of at least ``length + 1`` rows, in commit order, with
        the start law of ``load_episodes`` (``balance``); or ``indices=(episode_id, start)`` names the chunks.  Entries
        with no chunk (nothing eligible, or an index that names no held chunk) are zero rows with id and start -1;
        invalid indices are counted (``info()['invalid_requests']``) and ``check=True`` raises on them.  Asynchronous
        unless ``check``."""
        torch, env = self._torch, self.env
        if length is None or int(length) < 1:
            raise ValueError("length must be a positive number of rows")
        L = int(length)
        ids = starts = None
        if indices is not None:
            ids = torch.as_tensor(indices[0]).to(device=env.device, dtype=torch.int64).contiguous().reshape(-1)
            starts = torch.as_tensor(indices[1]).to(device=env.device, dtype=torch.int32).contiguous().reshape(-1)
            if ids.shape != starts.shape:
                raise ValueError("indices: episode_id and start must have the same length")
            if batch is not None and int(batch) != ids.numel():
                raise ValueError("batch does not match the number of indices")
            B = ids.numel()
        else:
            if batch is None:
                raise ValueError("batch is required when drawing")
            B = int(batch)
        out = {k: torch.empty((B, L) + self._spec[k][0], dtype=self._spec[k][1], device=env.device) for k in self.keys}
        out["episode_id"] = torch.empty(B, dtype=torch.int64, device=env.device)
        out["start"] = torch.empty(B, dtype=torch.int32, device=env.device)
        b = self._abi.RdStoreBatch()
        for k, f in (("lidar", "lidar_dev"), ("lidar_occupancy", "occupancy_dev"), ("pose", "pose_dev"),
                     ("velocity", "velocity_dev"), ("speed", "speed_dev"), ("action", "action_dev"),
                     ("reward", "reward_dev"), ("discount", "discount_dev"), ("progress", "progress_dev"),
                     ("time", "time_dev"), ("episode_id", "episode_id_dev"), ("start", "start_dev")):
            if k in out:
                setattr(b, f, out[k].data_ptr())
        before = self.info()["invalid_requests"] if check else 0
        with torch.cuda.device(env.device):
            env._check(env.lib.rd_store_sample(env._handle, B, L, int(bool(balance)),
                                                ids.data_ptr() if ids is not None else None,
                                                starts.data_ptr() if starts is not None else None,
                                                self._C.byref(b), env._stream()))
        if check:
            bad = self.info()["invalid_requests"] - before
            if bad:
                raise IndexError(f"{bad} of {B} requested chunks name no held episode rows (evicted id or start out of range)")
        return out

    # -- bookkeeping / export --
    def info(self) -> Dict[str, int]:
        """Synchronising: committed, held, held_rows, evicted, invalid_requests, draws, capacity_rows,
        max_episode_steps."""
        env = self.env
        s = self._abi.RdStoreSummary()
        with self._torch.cuda.device(env.device):
            env._check(env.lib.rd_store_info(env._handle, self._C.byref(s), None, 0, env._stream()))
        return s.as_dict()

    def held(self) -> np.ndarray:
        """(id, env, length) of the held episodes in commit order, int64 [held, 3]."""
        env, C = self.env, self._C
        n = self.info()["held"]
        arr = (self._abi.RdStoreEpisode * max(n, 1))()
        s = self._abi.RdStoreSummary()
        with self._torch.cuda.device(env.device):
            env._check(env.lib.rd_store_info(env._handle, C.byref(s), arr, n, env._stream()))
        return np.array([(e.id, e.env, e.length) for e in arr[:min(n, int(s.held))]], np.int64).reshape(-1, 3)

    def episodes(self, since_id: Optional[int] = None, max_rows_per_gather: int = 1 << 18) -> List[Dict[str, np.ndarray]]:
        """Host dicts of the held episodes (id >= since_id) in commit order, the format ``EpisodeRecorder`` hands to its
        callbacks.  Gathered on the device, episodes of one length at a time."""
        h = self.held()
        if since_id is not None:
            h = h[h[:, 0] >= int(since_id)]
        out: List[Optional[Dict[str, np.ndarray]]] = [None] * len(h)
        for length in np.unique(h[:, 2]):
            rows = np.flatnonzero(h[:, 2] == length)
            per = max(1, int(max_rows_per_gather) // int(length))
            for c0 in range(0, len(rows), per):
                sel = rows[c0:c0 + per]
                got = self.sample(length=int(length), indices=(h[sel, 0], np.zeros(len(sel), np.int32)))
                host = {k: got[k].cpu().numpy() for k in self.keys}
                for j, i in enumerate(sel):
                    out[i] = {k: host[k][j].copy() for k in self.keys}
        return out

    def save(self, directory, since_id: Optional[int] = None) -> List[pathlib.Path]:
        """``save_episodes`` of ``episodes(since_id)``: files ``load_episodes`` / ``count_episodes`` read."""
        return save_episodes(directory, self.episodes(since_id))
