"""GPU: the device-resident episode store (episodes.DeviceEpisodeStore over rd_store_*, csrc/rd_store.cuh).

* The committed episodes and every per-step returned dict equal, bit for bit, what EpisodeRecorder over HostSteppedEnv
  produces for the same config, seed and actions.
* Eviction follows the per-env ring rule; the sampler's draws equal the NumPy law of test_cpu_episode_store bit for
  bit, and its chunks equal slices of the exported episodes.
* Recorded rollouts of both on-device policies equal a Python loop of act() + store.step().
* save() writes files load_episodes / count_episodes read."""
import numpy as np
import pytest

from racing_dreamer_b200.episodes import (EpisodeRecorder, DeviceEpisodeStore, OBS_KEYS, count_episodes, load_episodes,
                                          max_episode_steps)
from test_cpu_episode_store import store_draw

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


def _config(**kw):
    from racing_dreamer_b200 import EnvConfig
    base = dict(n_envs=16, action_repeat=4, auto_reset=False, reset_mode="random", time_limit_steps=30, seed=11)
    base.update(kw)
    return EnvConfig(**base)


def _bitwise(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), (what, np.abs(a.astype(np.float64) - b.astype(np.float64)).max())


def _same_dict(host, dev, what):
    assert list(host) == list(dev), (what, list(host), list(dev))
    for k in host:
        _bitwise(host[k], dev[k].cpu().numpy() if hasattr(dev[k], "cpu") else dev[k], (what, k))


def _same_episodes(want, got):
    assert len(want) == len(got)
    for i, (w, g) in enumerate(zip(want, got)):
        assert list(w) == list(g), (i, list(w), list(g))
        for k in w:
            _bitwise(w[k], g[k], (i, k))


def _record_both(torch, ec, steps, precision=32, keep_obs=OBS_KEYS, capacity=None, seed=0, rng_seed=0):
    """Runs EpisodeRecorder(HostSteppedEnv) and DeviceEpisodeStore(BatchedRaceEnv) side by side on the same random
    actions, comparing the returned dicts every step.  Returns (recorder episodes, their envs, recorder, store)."""
    from racing_dreamer_b200 import BatchedRaceEnv
    from racing_dreamer_b200.host import HostSteppedEnv
    host = HostSteppedEnv(ec, device="cuda:0", n_shards=2)
    T = max_episode_steps(host.env.cfg)
    captured = []
    rec = EpisodeRecorder(host, max_len=T, callbacks=[captured.extend], precision=precision, keep_obs=keep_obs,
                          reset_mode=ec.reset_mode)
    env = BatchedRaceEnv(ec, device="cuda:0")
    store = DeviceEpisodeStore(env, capacity_rows=capacity or 4 * (T + 1), precision=precision, keep_obs=keep_obs,
                               reset_mode=ec.reset_mode, seed=seed)
    _same_dict(rec.reset(), store.reset(), "reset")
    rng = np.random.RandomState(rng_seed)
    envs = []
    A = max(1, ec.agents_per_world)
    for t in range(steps):
        a = rng.uniform(-1, 1, (ec.n_envs, 2)).astype(np.float32)
        out = rec.step(a)
        done = np.repeat(out["done"].reshape(-1, A).any(axis=1), A)
        envs.extend(np.flatnonzero(done).tolist())
        _same_dict(out, store.step(torch.from_numpy(a).cuda()), ("step", t))
    assert len(envs) == len(captured)
    host.close()
    return captured, envs, rec, store


CASES = {
    "two_tracks": dict(tracks=("austria", "columbia")),
    "occupancy": dict(tracks=("columbia",), obs_type="lidar_occupancy", n_envs=8),
    "precision16": dict(tracks=("austria",), precision=16),
    "normalize_lidar": dict(tracks=("austria",), normalize_lidar=True),
    "worlds_of_four": dict(tracks=("treitlstrasse_v2",), agents_per_world=4, reset_mode="random_ball"),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_store_equals_episode_recorder(torch_cuda, case):
    kw = dict(CASES[case])
    precision = kw.pop("precision", 32)
    captured, _, _, store = _record_both(torch_cuda, _config(**kw), steps=90, precision=precision)
    assert len(captured) >= 8, "the workload should end many episodes"
    _same_episodes(captured, store.episodes())
    info = store.info()
    assert info["committed"] == info["held"] == len(captured) and info["evicted"] == 0
    assert info["held_rows"] == sum(len(e["reward"]) for e in captured)
    store.env.close()


def test_eviction_follows_the_per_env_ring(torch_cuda):
    cap = 31     # time_limit_steps 30: the smallest ring the config allows
    captured, envs, rec, store = _record_both(torch_cuda, _config(tracks=("austria",), n_envs=8), steps=120, capacity=cap)
    head = np.zeros(8, np.int64)
    starts = []
    for ep, e in zip(captured, envs):   # rows of env e: its committed episodes back to back, then the one in progress
        starts.append(head[e])
        head[e] += len(ep["reward"])
    head += rec._len
    keep = [i for i, e in enumerate(envs) if starts[i] >= head[e] - cap]
    assert 0 < len(keep) < len(captured)
    _same_episodes([captured[i] for i in keep], store.episodes())
    assert np.array_equal(store.held()[:, 0], np.array(keep))
    info = store.info()
    assert info["committed"] == len(captured) and info["held"] == len(keep) and info["evicted"] == len(captured) - len(keep)
    store.env.close()


@pytest.mark.parametrize("seed", [0, 0x123456789ABCDEF])
def test_sampler(torch_cuda, seed):
    torch = torch_cuda
    captured, _, _, store = _record_both(torch, _config(tracks=("austria",)), steps=80, seed=seed, rng_seed=1)
    held = store.held()
    eps = store.episodes()
    call = 0
    for B, L, balance in ((50, 5, False), (64, 12, True), (7, 1, False), (33, 20, True), (50, 25, False)):
        got = store.sample(batch=B, length=L, balance=balance)
        want_id, want_start = store_draw(seed, call, B, L, held[:, [0, 2]], balance)
        call += 1
        ids, starts = got["episode_id"].cpu().numpy(), got["start"].cpu().numpy()
        _bitwise(want_id, ids, ("id", B, L, balance))
        _bitwise(want_start, starts, ("start", B, L, balance))
        if (ids < 0).all():
            continue
        pos = {int(i): j for j, i in enumerate(held[:, 0])}
        for b in range(B):
            ep = eps[pos[int(ids[b])]]
            for k in store.keys:
                _bitwise(ep[k][starts[b]:starts[b] + L], got[k][b].cpu().numpy(), (k, b))
        again = store.sample(length=L, indices=(got["episode_id"], got["start"]), check=True)
        for k in store.keys + ("episode_id", "start"):
            assert torch.equal(again[k], got[k]), k
    assert store.info()["draws"] == call
    # invalid explicit indices: never committed, negative id, start past the episode's end, chunk overrunning it
    n = len(captured)
    bad_ids = torch.tensor([n + 5, -3, int(held[0, 0]), int(held[0, 0])], dtype=torch.int64)
    bad_st = torch.tensor([0, 0, int(held[0, 2]), 1], dtype=torch.int32)
    before = store.info()["invalid_requests"]
    got = store.sample(length=int(held[0, 2]), indices=(bad_ids, bad_st))
    assert (got["episode_id"].cpu().numpy() == -1).all() and (got["start"].cpu().numpy() == -1).all()
    assert all(int(got[k].abs().sum() if got[k].dtype != torch.uint8 else got[k].sum()) == 0 for k in store.keys)
    assert store.info()["invalid_requests"] == before + 4
    with pytest.raises(IndexError):
        store.sample(length=3, indices=([n + 1], [0]), check=True)
    # longer than every episode: nothing eligible
    L = int(held[:, 2].max())
    got = store.sample(batch=5, length=L)
    assert (got["episode_id"].cpu().numpy() == -1).all() and float(got["reward"].abs().sum()) == 0.0
    store.env.close()


def _policy_pair(torch, kind, noise):
    from racing_dreamer_b200 import BatchedRaceEnv, DreamerPolicy, GapFollowerPolicy
    ec = _config(tracks=("austria",), n_envs=32, time_limit_steps=25, seed=4)
    pairs = []
    for _ in range(2):
        env = BatchedRaceEnv(ec, device="cuda:0")
        store = DeviceEpisodeStore(env, capacity_rows=400)
        pol = GapFollowerPolicy(env) if kind == "gap" else DreamerPolicy(env, "austria_dreamer", noise=noise)
        store.reset()
        pairs.append((env, store, pol))
    return pairs


@pytest.mark.parametrize("kind,noise", [("gap", None), ("dreamer", "zero"), ("dreamer", "philox")])
def test_recorded_rollout_equals_a_python_loop(torch_cuda, kind, noise):
    torch = torch_cuda
    (env1, s1, p1), (env2, s2, p2) = _policy_pair(torch, kind, noise)
    steps = 70
    if kind == "gap":
        p1.rollout(steps, store=s1)
    else:
        p1.rollout(steps, store=s1, noise=noise)
    for _ in range(steps):
        a = p2.act() if kind == "gap" else p2.act(noise=noise)
        s2.step(a)
    torch.cuda.synchronize()
    e1, e2 = s1.episodes(), s2.episodes()
    assert len(e1) >= 32
    _same_episodes(e2, e1)
    out1, out2 = s1._outputs(), s2._outputs()
    for k in out1:
        assert torch.equal(out1[k], out2[k]), k
    st = env1.read_stats()
    assert st["episodes"] == len(e1)
    ret = sum(float(np.sum(e["reward"], dtype=np.float64)) for e in e1)
    assert abs(ret - st["return_sum"]) <= 1e-4 * max(1.0, abs(st["return_sum"]))
    env1.close()
    env2.close()


def test_save_round_trips(torch_cuda, tmp_path):
    captured, _, _, store = _record_both(torch_cuda, _config(tracks=("austria",), n_envs=8), steps=50)
    first = int(store.held()[2, 0])
    paths = store.save(tmp_path, since_id=first)
    eps = store.episodes(since_id=first)
    assert len(paths) == len(eps) == len(captured) - 2
    assert count_episodes(tmp_path) == (len(eps), sum(len(e["reward"]) - 1 for e in eps))
    loaded = load_episodes(tmp_path, rescan=len(eps))
    key = lambda e: e["reward"].tobytes() + e["lidar"].tobytes()   # noqa: E731
    want = {key(e): e for e in eps}
    for _ in range(len(eps)):
        ep = next(loaded)
        w = want[key(ep)]
        for k in w:
            _bitwise(w[k], ep[k], k)
    store.env.close()


def test_construction_checks(torch_cuda):
    from racing_dreamer_b200 import BatchedRaceEnv
    env = BatchedRaceEnv(_config(tracks=("austria",), n_envs=4), device="cuda:0")
    T = max_episode_steps(env.cfg)
    assert T == 30
    with pytest.raises(RuntimeError, match="capacity_rows"):
        DeviceEpisodeStore(env, capacity_rows=T)
    store = DeviceEpisodeStore(env, capacity_rows=T + 1)
    assert store.info()["max_episode_steps"] == T     # the library's bound is the Python helper's
    # rd_store_sample refuses output buffers that overlap the caller's indices
    import ctypes as C
    from racing_dreamer_b200 import _abi
    ids = torch_cuda.zeros(4, dtype=torch_cuda.int64, device="cuda:0")
    st = torch_cuda.zeros(4, dtype=torch_cuda.int32, device="cuda:0")
    b = _abi.RdStoreBatch()
    b.episode_id_dev, b.start_dev = ids.data_ptr(), st.data_ptr()
    assert env.lib.rd_store_sample(env._handle, 4, 1, 0, ids.data_ptr(), st.data_ptr(), C.byref(b), None) != 0
    assert b"overlap" in env.lib.rd_last_error(env._handle)
    env.close()
    env = BatchedRaceEnv(_config(tracks=("austria",), n_envs=4, auto_reset=True), device="cuda:0")
    with pytest.raises(ValueError, match="auto_reset"):
        DeviceEpisodeStore(env, capacity_rows=100)
    env.close()
