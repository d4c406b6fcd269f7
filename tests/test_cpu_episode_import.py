"""CPU: the host side of importing episodes into the device episode store (episodes.DeviceEpisodeStore.insert / load).

* check_import: the checks every episode of a call passes before any device work.
* episode_files: sorted file order and shard selection; npz_meta: shapes and dtypes from the .npy headers.
* imported_held against a row-by-row simulation of the import arena and its table of import_capacity_rows + 1 slots.
* the draw law over the eligible list imported-then-recorded (store_draw of test_cpu_episode_store)."""
import numpy as np
import pytest

from racing_dreamer_b200.episodes import check_import, episode_files, imported_held, npz_meta, save_episodes
from test_cpu_episode_store import store_draw

ID0 = 1 << 62
ROWS = {"lidar": (8,), "pose": (6,), "speed": (), "lidar_occupancy": (64, 64, 1), "action": (2,), "reward": ()}


def _episode(n, dtype=np.float32, **over):
    ep = {k: np.zeros((n,) + s, np.uint8 if k == "lidar_occupancy" else dtype) for k, s in ROWS.items()}
    ep.update(over)
    return ep


def _meta(ep):
    return {k: (np.shape(v), np.asarray(v).dtype) for k, v in ep.items()}


def test_check_import_accepts_and_returns_lengths():
    eps = [_episode(5), _episode(1, np.float16), _episode(7, np.float64, extra=np.zeros(3, np.int64))]
    assert check_import([_meta(e) for e in eps], ROWS, 7) == [5, 1, 7]


@pytest.mark.parametrize("bad,match", [
    (dict(reward=None), "missing"),
    (dict(reward=np.zeros(4, np.float32)), "common length"),
    (dict(lidar=np.zeros((5, 9), np.float32)), "shape"),
    (dict(lidar_occupancy=np.zeros((5, 64, 64), np.uint8)), "shape"),
    (dict(pose=np.zeros((5, 6), np.int32)), "float16"),
    (dict(lidar_occupancy=np.zeros((5, 64, 64, 1), np.float32)), "uint8"),
    (dict(speed=np.zeros(5, np.complex64)), "float16"),
])
def test_check_import_rejects(bad, match):
    ep = _episode(5)
    for k, v in bad.items():
        if v is None:
            del ep[k]
        else:
            ep[k] = v
    with pytest.raises(ValueError, match=match):
        check_import([_meta(_episode(3)), _meta(ep)], ROWS, 100)


def test_check_import_rejects_empty_and_too_long():
    with pytest.raises(ValueError, match="common length"):
        check_import([_meta(_episode(0))], ROWS, 10)
    with pytest.raises(ValueError, match="import_capacity_rows"):
        check_import([_meta(_episode(11))], ROWS, 10)
    with pytest.raises(ValueError, match="episode 1"):
        check_import([_meta(_episode(3)), _meta(_episode(11))], ROWS, 10)


def test_episode_files_order_and_shards(tmp_path):
    paths = save_episodes(tmp_path, [_episode(n) for n in (3, 4, 5, 6, 7)])
    (tmp_path / "notes.txt").write_text("not an episode")
    files = episode_files(tmp_path)
    assert files == sorted(paths)
    for world in (1, 2, 3, 7):
        shards = [episode_files(tmp_path, (r, world)) for r in range(world)]
        assert sorted(sum(shards, [])) == files
        for r, s in enumerate(shards):
            assert s == [f for i, f in enumerate(files) if i % world == r]
    with pytest.raises(ValueError):
        episode_files(tmp_path, (2, 2))


def test_npz_meta_reads_headers(tmp_path):
    [path] = save_episodes(tmp_path, [_episode(9, np.float16, extra=np.zeros(2))])
    meta = npz_meta(path, list(ROWS) + ["missing"])
    assert meta == {k: ((9,) + s, np.dtype(np.uint8 if k == "lidar_occupancy" else np.float16)) for k, s in ROWS.items()}
    bad = tmp_path / "broken.npz"
    bad.write_bytes(path.read_bytes()[:100])
    with pytest.raises(Exception):
        npz_meta(bad, list(ROWS))


def _simulate_arena(calls, cap):
    """Row by row: the ring's owner of every slot and a table of cap + 1 slots indexed by k mod (cap + 1), written for
    every imported episode k.  Returns (held by ownership of all rows, held by the table rule) over all episodes."""
    owner = np.full(cap, -1, np.int64)          # (episode << 20) | row of the slot's content
    table = np.full(cap + 1, -1, np.int64)
    start, length = [], []
    head = k = 0
    for lengths in calls:
        for n in lengths:
            table[k % (cap + 1)] = k
            start.append(head)
            length.append(n)
            for r in range(n):
                owner[(head + r) % cap] = (k << 20) | r
            head += n
            k += 1
    by_rows = np.array([all(owner[(start[i] + r) % cap] == (i << 20) | r for r in range(length[i])) for i in range(k)])
    by_table = np.array([table[i % (cap + 1)] == i and start[i] >= head - cap for i in range(k)])
    return by_rows, by_table


@pytest.mark.parametrize("seed", range(6))
def test_arena_holds_what_the_oracle_says(seed):
    rng = np.random.RandomState(seed)
    cap = int(rng.randint(1, 40))
    calls = [list(rng.randint(1, cap + 1, size=rng.randint(0, 12))) for _ in range(rng.randint(1, 8))]
    if seed == 0:
        cap, calls = 5, [[1] * 13, [5], [2, 1]]     # many one-row episodes: the table wraps within a call
    by_rows, by_table = _simulate_arena(calls, cap)
    flat = sum(calls, [])
    assert np.array_equal(by_rows, by_table)
    assert np.array_equal(imported_held(flat, cap), by_rows)
    # what one call keeps of its own episodes is the same rule on the call's lengths (the host stages only those)
    for lengths in calls:
        if lengths:
            assert np.array_equal(imported_held(lengths, cap), _simulate_arena([lengths], cap)[0])


def test_draw_law_over_imported_then_recorded():
    imported = [(ID0 + k, n) for k, n in enumerate((40, 8, 25))]
    recorded = [(0, 30), (1, 12), (2, 60)]
    for call in range(4):
        # imported episodes too short for the length leave the recorded-only draws as they are
        a = store_draw(7, call, 256, 10, recorded)
        b = store_draw(7, call, 256, 10, [(ID0, 10), (ID0 + 1, 3)] + recorded)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    ids = np.concatenate([store_draw(7, k, 4096, 10, imported + recorded)[0] for k in range(4)])
    elig = [i for i, n in imported + recorded if n >= 11]
    assert set(np.unique(ids)) == set(elig)
    counts = np.array([(ids == i).sum() for i in elig])
    from scipy import stats
    assert stats.chisquare(counts).pvalue > 1e-3
    # the list is imported-then-recorded: index j of the concatenated eligible list
    x = store_draw(3, 0, 64, 10, imported + recorded)[0]
    y = store_draw(3, 0, 64, 10, recorded + imported)[0]
    assert not np.array_equal(x, y)
