"""GPU: importing episodes into the device episode store (DeviceEpisodeStore.insert / load, rd_store_import*).

* Round trip: save() then load() into a fresh store gives the files back bit for bit, at precision 32 and 16 and with
  lidar_occupancy, and the store samples at once.
* Conversion of float16/32/64 inputs equals episodes._convert (numpy astype).
* Draws over imported and recorded episodes equal the NumPy law with the list imported-then-recorded; chunks are
  slices of the exported episodes; explicit indices take imported ids; evicted ones give zero rows and -1.
* The arena holds the episodes imported_held says; recording after an import is unchanged; rejected calls import
  nothing; shards of one directory partition it."""
import numpy as np
import pytest

from racing_dreamer_b200.episodes import (DeviceEpisodeStore, EpisodeRecorder, _convert, episode_files,
                                          imported_held, max_episode_steps)
from test_cpu_episode_store import store_draw
from test_gpu_episode_store import _bitwise, _config, _record_both, _same_dict, _same_episodes

pytestmark = pytest.mark.gpu
ID0 = DeviceEpisodeStore.IMPORTED_ID0


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


def _fresh(ec, precision=32, import_rows=2000, seed=0, capacity=None):
    from racing_dreamer_b200 import BatchedRaceEnv
    env = BatchedRaceEnv(ec, device="cuda:0")
    T = max_episode_steps(env.cfg)
    return DeviceEpisodeStore(env, capacity_rows=capacity or 4 * (T + 1), precision=precision, reset_mode=ec.reset_mode,
                              seed=seed, import_capacity_rows=import_rows)


def _synthetic(store, lengths, dtype, rng):
    """Episodes of the store's keys with values that exercise rounding: wide magnitudes, half subnormals, overflow."""
    eps = []
    for n in lengths:
        ep = {}
        for k in store.keys:
            shape = (n,) + store._spec[k][0]
            if k == "lidar_occupancy":
                ep[k] = rng.randint(0, 256, size=shape).astype(np.uint8)
            else:
                v = rng.standard_normal(shape) * 10.0 ** rng.randint(-8, 6, size=shape)
                ep[k] = v.astype(dtype)
        eps.append(ep)
    return eps


@pytest.mark.parametrize("case", ["precision32", "precision16", "occupancy"])
def test_save_then_load_round_trips(torch_cuda, tmp_path, case):
    kw = dict(tracks=("columbia",), obs_type="lidar_occupancy", n_envs=8) if case == "occupancy" else dict(tracks=("austria",))
    precision = 16 if case == "precision16" else 32
    ec = _config(**kw)
    captured, _, _, store = _record_both(torch_cuda, ec, steps=60, precision=precision)
    paths = store.save(tmp_path)
    assert len(paths) == len(captured)
    store.env.close()
    fresh = _fresh(ec, precision=precision)
    ids = fresh.load(tmp_path)
    assert np.array_equal(ids, ID0 + np.arange(len(paths)))
    want = [dict(np.load(p)) for p in sorted(paths)]
    _same_episodes(want, fresh.episodes(imported=True))
    held = fresh.held(imported=True)
    assert np.array_equal(held[:, 0], ids) and (held[:, 1] == -1).all()
    assert np.array_equal(held[:, 2], [len(e["reward"]) for e in want])
    info = fresh.info()
    assert info["imported"] == info["imported_held"] == len(want) and info["imported_evicted"] == 0
    assert info["imported_rows"] == sum(len(e["reward"]) for e in want)
    assert info["committed"] == info["held"] == 0 and fresh.episodes() == []
    # a resumed learner samples before any reset or step
    got = fresh.sample(batch=16, length=5)
    assert (got["episode_id"].cpu().numpy() >= ID0).all()
    fresh.env.close()


@pytest.mark.parametrize("precision,dtype", [(16, np.float32), (32, np.float16), (16, np.float64), (32, np.float64),
                                             (16, np.float16), (32, np.float32)])
def test_conversion_equals_convert(torch_cuda, precision, dtype):
    store = _fresh(_config(tracks=("austria",), n_envs=4), precision=precision)
    eps = _synthetic(store, [3, 17, 1], dtype, np.random.RandomState(precision + np.dtype(dtype).itemsize))
    store.insert(eps)
    got = store.episodes(imported=True)
    _same_episodes([{k: _convert(e[k], precision) for k in store.keys} for e in eps], got)
    store.env.close()


def test_mixed_sampling(torch_cuda):
    torch = torch_cuda
    ec = _config(tracks=("austria",))
    mixed = _fresh(ec, seed=0x5EED, import_rows=600)
    rng = np.random.RandomState(2)
    imp = _synthetic(mixed, [40, 3, 25, 31, 12, 60], np.float32, rng)
    mixed.insert(imp[:4])
    mixed.reset()
    a = np.random.RandomState(9)
    for _ in range(60):
        mixed.step(torch.from_numpy(a.uniform(-1, 1, (ec.n_envs, 2)).astype(np.float32)).cuda())
    mixed.insert(imp[4:])
    held_rec, held_imp = mixed.held(), mixed.held(imported=True)
    assert len(held_rec) >= 8 and len(held_imp) == 6
    both = np.concatenate([held_imp, held_rec])
    eps = mixed.episodes(imported=True) + mixed.episodes()
    pos = {int(i): j for j, i in enumerate(both[:, 0])}
    drawn = []
    for call, (B, L, balance) in enumerate(((50, 5, False), (64, 12, True), (33, 20, False), (50, 30, True))):
        got = mixed.sample(batch=B, length=L, balance=balance)
        want_id, want_start = store_draw(0x5EED, call, B, L, both[:, [0, 2]], balance)
        ids, starts = got["episode_id"].cpu().numpy(), got["start"].cpu().numpy()
        _bitwise(want_id, ids, ("id", B, L))
        _bitwise(want_start, starts, ("start", B, L))
        drawn.extend(ids.tolist())
        for b in range(B):
            for k in mixed.keys:
                _bitwise(eps[pos[int(ids[b])]][k][starts[b]:starts[b] + L], got[k][b].cpu().numpy(), (k, b))
    assert min(drawn) < ID0 <= max(drawn)
    # explicit indices on imported ids, with the imported rows converted as _convert does
    got = mixed.sample(length=3, indices=(held_imp[:, 0], np.full(len(held_imp), 0, np.int32)), check=True)
    for j, ep in enumerate(imp):
        for k in mixed.keys:
            _bitwise(_convert(ep[k][:3], 32), got[k][j].cpu().numpy(), (k, j))
    mixed.env.close()


def test_arena_eviction_and_invalid_imported_ids(torch_cuda):
    torch = torch_cuda
    cap = 50
    store = _fresh(_config(tracks=("austria",), n_envs=4), import_rows=cap)
    rng = np.random.RandomState(5)
    calls = [[10, 20], [1] * 8, [30, 5, 7, 50, 4], [3] * 25, [12, 1]]   # the third and fourth calls exceed the arena
    eps, ids = [], []
    for lengths in calls:
        e = _synthetic(store, lengths, np.float32, rng)
        ids.extend(store.insert(e).tolist())
        eps.extend(e)
        flat = [len(x["reward"]) for x in eps]
        keep = np.flatnonzero(imported_held(flat, cap))
        assert np.array_equal(store.held(imported=True)[:, 0], ID0 + keep)
        _same_episodes([{k: eps[i][k] for k in store.keys} for i in keep], store.episodes(imported=True))
        info = store.info()
        assert info["imported"] == len(eps) and info["imported_held"] == len(keep)
        assert info["imported_evicted"] == len(eps) - len(keep)
    assert ids == (ID0 + np.arange(len(eps))).tolist()
    # evicted, never imported and out-of-range imported requests: zero rows, id / start -1, counted
    keep_ids = store.held(imported=True)
    bad_ids = torch.tensor([ID0, ID0 + len(eps) + 3, int(keep_ids[0, 0]), ID0 - 1], dtype=torch.int64)
    bad_st = torch.tensor([0, 0, int(keep_ids[0, 2]), 0], dtype=torch.int32)
    before = store.info()["invalid_requests"]
    got = store.sample(length=1, indices=(bad_ids, bad_st))
    assert (got["episode_id"].cpu().numpy() == -1).all() and (got["start"].cpu().numpy() == -1).all()
    assert all(float(got[k].abs().sum()) == 0.0 for k in store.keys)
    assert store.info()["invalid_requests"] == before + 4
    with pytest.raises(IndexError):
        store.sample(length=1, indices=([ID0], [0]), check=True)
    store.env.close()


def test_recording_after_an_import(torch_cuda, tmp_path):
    from racing_dreamer_b200.host import HostSteppedEnv
    torch = torch_cuda
    ec = _config(tracks=("austria",), n_envs=8)
    store = _fresh(ec, import_rows=300)
    imp = _synthetic(store, [30, 7, 100], np.float32, np.random.RandomState(1))
    store.insert(imp)
    host = HostSteppedEnv(ec, device="cuda:0", n_shards=2)
    captured = []
    rec = EpisodeRecorder(host, max_len=max_episode_steps(host.env.cfg), callbacks=[captured.extend],
                          reset_mode=ec.reset_mode)
    _same_dict(rec.reset(), store.reset(), "reset")
    rng = np.random.RandomState(0)
    for t in range(50):
        a = rng.uniform(-1, 1, (ec.n_envs, 2)).astype(np.float32)
        _same_dict(rec.step(a), store.step(torch.from_numpy(a).cuda()), ("step", t))
    host.close()
    assert len(captured) >= 8
    _same_episodes(captured, store.episodes())
    assert np.array_equal(store.held()[:, 0], np.arange(len(captured)))
    paths = store.save(tmp_path)
    assert len(paths) == len(captured) == len(episode_files(tmp_path))
    info = store.info()
    assert info["imported"] == info["imported_held"] == 3 and info["committed"] == len(captured)
    store.env.close()


def test_rejected_imports_change_nothing(torch_cuda, tmp_path):
    store = _fresh(_config(tracks=("austria",), n_envs=4), import_rows=40)
    rng = np.random.RandomState(3)
    store.insert(_synthetic(store, [5, 6], np.float32, rng))
    before = store.info()
    good = _synthetic(store, [4], np.float32, rng)[0]
    bads = [{k: v for k, v in good.items() if k != "pose"},
            dict(good, reward=good["reward"][:3]),
            dict(good, lidar=good["lidar"][:, :-1]),
            dict(good, action=good["action"].astype(np.int32)),
            _synthetic(store, [41], np.float32, rng)[0],
            {k: v[:0] for k, v in good.items()}]
    for bad in bads:
        with pytest.raises(ValueError):
            store.insert([good, bad])
        assert store.info() == before
    store.insert([dict(good, extra=np.zeros(4))])     # extra keys are ignored
    assert store.info()["imported"] == before["imported"] + 1
    # an unreadable file is skipped with a message; the others import
    from racing_dreamer_b200.episodes import save_episodes
    paths = save_episodes(tmp_path, [good, good])
    paths[0].write_bytes(b"not a zip file")
    assert len(store.load(tmp_path)) == 1
    store.env.close()
    plain = _fresh(_config(tracks=("austria",), n_envs=4), import_rows=0)
    with pytest.raises(ValueError, match="import arena"):
        plain.insert([good])
    info = plain.info()
    assert info["import_capacity_rows"] == 0 and info["imported"] == 0
    plain.env.close()


def test_shards_partition_a_directory(torch_cuda, tmp_path):
    from racing_dreamer_b200.episodes import save_episodes
    ec = _config(tracks=("austria",), n_envs=4)
    ref = _fresh(ec)
    eps = _synthetic(ref, list(range(3, 14)), np.float32, np.random.RandomState(4))
    save_episodes(tmp_path, eps)
    want = [dict(np.load(p)) for p in episode_files(tmp_path)]
    ref.env.close()
    got = []
    for rank in range(2):
        store = _fresh(ec)
        ids = store.load(tmp_path, shard=(rank, 2))
        assert len(ids) == len(want[rank::2])
        _same_episodes([{k: e[k] for k in store.keys} for e in want[rank::2]], store.episodes(imported=True))
        got.extend(store.episodes(imported=True))
        store.env.close()
    assert len(got) == len(want)
