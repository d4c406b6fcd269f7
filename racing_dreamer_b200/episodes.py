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
import os
import pathlib
import uuid
import zipfile
from concurrent.futures import ThreadPoolExecutor
from typing import Callable, Dict, Iterator, List, Optional, Sequence, Tuple

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


def episode_files(directory, shard: Optional[Tuple[int, int]] = None) -> List[pathlib.Path]:
    """The ``*.npz`` files of `directory` in sorted order (``load_episodes``' order); ``shard=(rank, world)`` keeps those
    whose index in that order is ``rank`` modulo ``world``, so that the ranks of one run split a directory."""
    files = sorted(pathlib.Path(directory).expanduser().glob("*.npz"))
    if shard is None:
        return files
    rank, world = (int(v) for v in shard)
    if world < 1 or not 0 <= rank < world:
        raise ValueError(f"shard {shard}: expected (rank, world) with 0 <= rank < world")
    return files[rank::world]


def npz_meta(path, keys: Sequence[str]) -> Dict[str, Tuple[tuple, np.dtype]]:
    """(shape, dtype) of the arrays `keys` of an ``.npz`` file, read from the ``.npy`` headers without decompressing
    the data; keys the file lacks are left out.  Raises on a file that is not a readable archive."""
    from numpy.lib import format as npf
    readers = {(1, 0): npf.read_array_header_1_0, (2, 0): npf.read_array_header_2_0}
    out = {}
    with zipfile.ZipFile(path) as z:
        names = set(z.namelist())
        for k in keys:
            if k + ".npy" not in names:
                continue
            with z.open(k + ".npy") as f:
                version = npf.read_magic(f)
                if version in readers:
                    shape, _, dtype = readers[version](f)
                else:       # a newer header format: decode the array
                    a = npf.read_array(f)
                    shape, dtype = a.shape, a.dtype
            out[k] = (tuple(shape), np.dtype(dtype))
    return out


_FLOAT_DTYPES = (np.dtype(np.float16), np.dtype(np.float32), np.dtype(np.float64))


def check_import(metas: Sequence[Dict[str, Tuple[tuple, np.dtype]]], row_shapes: Dict[str, tuple],
                 capacity_rows: int, names: Optional[Sequence[str]] = None) -> List[int]:
    """Lengths of the episodes described by `metas` (key -> (shape, dtype)), or ValueError naming the first episode a
    ``DeviceEpisodeStore`` with these row shapes and import arena cannot take: a missing key, keys of different
    lengths or of no rows, a row shape other than the store's, a float key that is not float16/32/64, a
    ``lidar_occupancy`` that is not uint8, or more rows than the arena holds.  Extra keys are ignored."""
    lengths = []
    for i, meta in enumerate(metas):
        what = names[i] if names is not None else f"episode {i}"
        missing = [k for k in row_shapes if k not in meta]
        if missing:
            raise ValueError(f"{what}: missing keys {missing}")
        n = {meta[k][0][0] if len(meta[k][0]) else None for k in row_shapes}
        if len(n) != 1 or None in n or min(n) < 1:
            raise ValueError(f"{what}: the keys need one common length of at least one row, got "
                             f"{ {k: meta[k][0] for k in row_shapes} }")
        length = n.pop()
        for k, row in row_shapes.items():
            shape, dtype = meta[k]
            if tuple(shape[1:]) != tuple(row):
                raise ValueError(f"{what}: '{k}' rows have shape {tuple(shape[1:])}, the store's are {tuple(row)}")
            if k == "lidar_occupancy" and dtype != np.uint8:
                raise ValueError(f"{what}: 'lidar_occupancy' is {dtype}, expected uint8")
            if k != "lidar_occupancy" and dtype not in _FLOAT_DTYPES:
                raise ValueError(f"{what}: '{k}' is {dtype}, expected float16, float32 or float64")
        if length > capacity_rows:
            raise ValueError(f"{what}: {length} rows exceed import_capacity_rows = {capacity_rows}")
        lengths.append(int(length))
    return lengths


def imported_held(lengths: Sequence[int], capacity_rows: int) -> np.ndarray:
    """Which of the episodes imported in this order, with these lengths, an import arena of `capacity_rows` rows holds:
    those whose first row has not been overwritten by the rows imported after it."""
    lengths = np.asarray(lengths, np.int64)
    first = np.cumsum(lengths) - lengths
    return first >= lengths.sum() - int(capacity_rows)


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
    ``capacity_rows`` must exceed ``max_episode_steps(env.cfg)``.  ``seed`` keys the sampler's Philox stream.

    ``import_capacity_rows > 0`` adds an import arena of that many rows (same row format and precision), which
    ``insert`` / ``load`` fill with episodes from outside the store -- saved files of this or another run, the
    reference's own episodes -- so that a resumed learner samples what it saved.  Imported episode k gets id
    ``IMPORTED_ID0 + k`` and is held while its first row has not been overwritten; importing past the arena's end evicts
    the oldest imported episodes.  Draws pick from the held imported episodes in import order, then the held recorded
    ones in commit order.  Imports never touch the recording: ``reset()`` keeps imported episodes, and ``episodes()``,
    ``held()`` and ``save()`` leave them out unless asked with ``imported=True``."""

    IMPORTED_ID0 = 1 << 62
    _IMPORT_CHUNK_BYTES = 64 << 20    # staged bytes per device import (two such buffers, pinned and on the device)

    def __init__(self, env, capacity_rows: int, precision: int = 32, keep_obs: Sequence[str] = OBS_KEYS,
                 reset_mode: Optional[str] = None, seed: int = 0, import_capacity_rows: int = 0):
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
        self.import_capacity_rows = int(import_capacity_rows)
        if self.import_capacity_rows < 0:
            raise ValueError("import_capacity_rows must be >= 0")
        self._stage = None
        with torch.cuda.device(env.device):
            env._check(env.lib.rd_store_init(env._handle, C.byref(sc)))
            if self.import_capacity_rows:
                env._check(env.lib.rd_store_import_init(env._handle, self.import_capacity_rows))

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
        ``start`` i32 [B].  Drawn uniformly over the held episodes of at least ``length + 1`` rows -- imported ones in
        import order, then recorded ones in commit order -- with the start law of ``load_episodes`` (``balance``); or
        ``indices=(episode_id, start)`` names the chunks (recorded or imported ids).  Entries
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
        max_episode_steps (recorded episodes), and imported, imported_held, imported_rows, imported_evicted,
        import_capacity_rows (the import arena)."""
        env = self.env
        s = self._abi.RdStoreSummary()
        si = self._abi.RdStoreImportSummary()
        with self._torch.cuda.device(env.device):
            env._check(env.lib.rd_store_info(env._handle, self._C.byref(s), None, 0, env._stream()))
            env._check(env.lib.rd_store_import_info(env._handle, self._C.byref(si), None, 0, env._stream()))
        out = s.as_dict()
        i = si.as_dict()
        out.update(imported=i["imported"], imported_held=i["held"], imported_rows=i["held_rows"],
                   imported_evicted=i["evicted"], import_capacity_rows=i["capacity_rows"])
        return out

    def held(self, imported: bool = False) -> np.ndarray:
        """(id, env, length) of the held episodes in commit order, int64 [held, 3]; ``imported=True``: of the held
        imported episodes in import order (env -1)."""
        env, C, abi = self.env, self._C, self._abi
        fn, summary = ((env.lib.rd_store_import_info, abi.RdStoreImportSummary) if imported else
                       (env.lib.rd_store_info, abi.RdStoreSummary))
        n = self.info()["imported_held" if imported else "held"]
        arr = (abi.RdStoreEpisode * max(n, 1))()
        s = summary()
        with self._torch.cuda.device(env.device):
            env._check(fn(env._handle, C.byref(s), arr, n, env._stream()))
        return np.array([(e.id, e.env, e.length) for e in arr[:min(n, int(s.held))]], np.int64).reshape(-1, 3)

    def episodes(self, since_id: Optional[int] = None, max_rows_per_gather: int = 1 << 18,
                 imported: bool = False) -> List[Dict[str, np.ndarray]]:
        """Host dicts of the held episodes (id >= since_id) in commit order, the format ``EpisodeRecorder`` hands to its
        callbacks; ``imported=True``: of the held imported episodes in import order.  Gathered on the device, episodes
        of one length at a time."""
        h = self.held(imported)
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
        """``save_episodes`` of ``episodes(since_id)``: files ``load_episodes`` / ``count_episodes`` read.  Imported
        episodes are not written again (after a resume they are on disk already)."""
        return save_episodes(directory, self.episodes(since_id))

    # -- import --
    def _row_shapes(self) -> Dict[str, tuple]:
        return {k: self._spec[k][0] for k in self.keys}

    def insert(self, episodes: Sequence[Dict[str, np.ndarray]]) -> np.ndarray:
        """Imports episode dicts -- those ``EpisodeRecorder`` hands to its callbacks, ``episodes()`` returns or
        ``dict(np.load(file))`` reads -- into the import arena; returns their ids (int64, in order).

        Every kept key must be present (others are ignored), all with one length of 1 to ``import_capacity_rows`` rows,
        the store's row shapes, float16/32/64 floats and uint8 ``lidar_occupancy``.  All episodes are checked before any
        device work, so a call that raises ``ValueError`` imports nothing.  Rows are converted on the device to the
        store's precision exactly as ``_convert`` does (numpy ``astype``).  Whether the observations were normalised as
        the env's are (``normalize_lidar``, the baselines' normalisation) cannot be told from the data and is not
        checked.  Asynchronous: the arrays are copied before it returns."""
        episodes = list(episodes)
        metas = [{k: (np.shape(v), np.asarray(v).dtype) for k, v in ep.items() if k in self.keys} for ep in episodes]
        lengths = self._check_import(metas)
        return self._import(lengths, [lambda ep=ep: ep for ep in episodes])

    def load(self, directory, shard: Optional[Tuple[int, int]] = None, workers: Optional[int] = None) -> np.ndarray:
        """Imports the ``*.npz`` episodes of `directory` in sorted file order (``load_episodes``' order), as ``insert``
        does; ``shard=(rank, world)`` takes the files whose index in that order is ``rank`` modulo ``world``.  A file
        that cannot be read is skipped with a message, as ``load_episodes`` does.  The files' headers are checked
        before any device work; their data is decompressed on `workers` threads, overlapped with the copies to the
        device, and files the arena would not hold at the end of the call are not decompressed.  Returns the ids."""
        paths, metas = [], []
        for path in episode_files(directory, shard):
            try:
                metas.append(npz_meta(path, self.keys))
            except Exception as e:  # noqa: BLE001 - a half-written file must not stop training (reference behaviour)
                print(f"Could not load episode: {e}")
                continue
            paths.append(path)
        lengths = self._check_import(metas, [str(p) for p in paths])
        keys = self.keys

        def read(path):
            try:
                with np.load(path) as z:
                    return {k: z[k] for k in keys}
            except Exception as e:  # noqa: BLE001
                print(f"Could not load episode: {e}")
                return None
        workers = int(workers or min(8, os.cpu_count() or 1))
        with ThreadPoolExecutor(max_workers=workers) as pool:
            return self._import(lengths, [lambda p=p: read(p) for p in paths], pool, 2 * workers)

    def _check_import(self, metas, names=None) -> List[int]:
        if self.import_capacity_rows == 0:
            raise ValueError("this store has no import arena: create it with import_capacity_rows > 0")
        return check_import(metas, self._row_shapes(), self.import_capacity_rows, names)

    def _import(self, lengths: List[int], readers, pool=None, ahead: int = 1) -> np.ndarray:
        """Registers the episodes the arena will not hold after the call without their data, then stages the others in
        chunks of up to _IMPORT_CHUNK_BYTES (one element type per key and chunk) through two pinned buffers, each
        chunk's copy and k_store_import enqueued on the current stream.  readers[i]() -> the dict of episode i, or None
        (skipped).  With a pool, up to `ahead` readers run ahead of the staging."""
        torch, env, C = self._torch, self.env, self._C
        n_before = self.info()["imported"]
        keep = imported_held(lengths, self.import_capacity_rows) if lengths else np.zeros(0, bool)
        n_drop = int(np.argmax(keep)) if keep.any() else len(lengths)
        registered = []                              # indices of the episodes imported, in order
        with torch.cuda.device(env.device):
            if n_drop:
                lens = (C.c_int32 * n_drop)(*lengths[:n_drop])
                env._check(env.lib.rd_store_import(env._handle, n_drop, lens, None, env._stream()))
                registered.extend(range(n_drop))
            todo = list(range(n_drop, len(lengths)))
            if pool is None:
                results = ((i, readers[i]()) for i in todo)
            else:
                def results():
                    futs = {}
                    for j, i in enumerate(todo):
                        for i2 in todo[j:j + ahead]:
                            if i2 not in futs:
                                futs[i2] = pool.submit(readers[i2])
                        yield i, futs.pop(i).result()
                results = results()
            chunk, chunk_bytes, chunk_types = [], 0, None
            for i, ep in results:
                if ep is None:
                    continue
                arrs = {k: np.ascontiguousarray(ep[k]) for k in self.keys}
                types = tuple(arrs[k].dtype for k in self.keys)
                nbytes = sum(a.nbytes + 16 for a in arrs.values())
                if chunk and (types != chunk_types or chunk_bytes + nbytes > self._IMPORT_CHUNK_BYTES):
                    self._stage_chunk(chunk)
                    chunk, chunk_bytes = [], 0
                chunk.append(arrs)
                chunk_bytes += nbytes
                chunk_types = types
                registered.append(i)
            if chunk:
                self._stage_chunk(chunk)
        return self.IMPORTED_ID0 + n_before + np.arange(len(registered), dtype=np.int64)

    def _stage_chunk(self, chunk: List[Dict[str, np.ndarray]]) -> None:
        torch, env, C, abi = self._torch, self.env, self._C, self._abi
        offs, total = {}, 0
        for k in self.keys:
            offs[k] = total
            total += -(-sum(ep[k].nbytes for ep in chunk) // 16) * 16
        if self._stage is None or self._stage["host"][0].numel() < total:
            for ev in (self._stage or {}).get("done", ()):
                if ev is not None:
                    ev.synchronize()
            size = max(total, self._IMPORT_CHUNK_BYTES)
            self._stage = {"host": [torch.empty(size, dtype=torch.uint8, pin_memory=True) for _ in range(2)],
                           "dev": [torch.empty(size, dtype=torch.uint8, device=env.device) for _ in range(2)],
                           "done": [None, None], "next": 0}
        st = self._stage
        b = st["next"]
        st["next"] ^= 1
        if st["done"][b] is not None:
            st["done"][b].synchronize()              # the previous copy out of this pinned buffer has run
        host, dev = st["host"][b], st["dev"][b]
        hnp = host.numpy()
        for k in self.keys:
            o = offs[k]
            for ep in chunk:
                a = ep[k]
                hnp[o:o + a.nbytes] = a.reshape(-1).view(np.uint8)
                o += a.nbytes
        dev[:total].copy_(host[:total], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        st["done"][b] = ev
        rows = abi.RdStoreImportRows()
        field = {"lidar_occupancy": "occupancy"}
        for k in self.keys:
            f = field.get(k, k)
            setattr(rows, f + "_dev", dev.data_ptr() + offs[k])
            setattr(rows, f + "_type", chunk[0][k].dtype.itemsize)
        lens = (C.c_int32 * len(chunk))(*[len(ep["reward"]) for ep in chunk])
        env._check(env.lib.rd_store_import(env._handle, len(chunk), lens, C.byref(rows), env._stream()))
