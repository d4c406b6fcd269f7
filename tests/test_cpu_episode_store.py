"""CPU: the draw law of the device-resident episode store (csrc/rd_store.cuh k_store_draw), restated in NumPy, and the
capacity bound of a store (episodes.max_episode_steps).

Philox4x32-10 is checked against Random123's published known-answer vectors and against the oracle's own
philox4x32_10 (oracle/rd_oracle.c, compiled here from its source).  The GPU tests compare the kernel's draws with
``store_draw`` bit for bit."""
import ctypes as C
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest
from scipy import stats

from racing_dreamer_b200 import _abi
from racing_dreamer_b200.episodes import max_episode_steps

ROOT = Path(__file__).resolve().parents[1]
STREAM_STORE = 0x53544F52     # RD_STREAM_STORE
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10 (counter words as arrays, key words as ints) -> four uint32 arrays."""
    c = [np.asarray(x, np.uint64) & _MASK for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0 & 0xFFFFFFFF), np.uint64(k1 & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
        k0 = (k0 + np.uint64(0x9E3779B9)) & _MASK
        k1 = (k1 + np.uint64(0xBB67AE85)) & _MASK
    return [x.astype(np.uint32) for x in c]


def store_draw(seed, call, batch, length, held, balance=False):
    """(episode_id i64 [B], start i32 [B]) of drawing sample call `call` of a store with sampler seed `seed`.

    held: (id, length) of the held episodes in commit order.  Entry b: Philox4x32-10 with key (seed_lo, seed_hi ^
    RD_STREAM_STORE) and counter (b, call, 0, 0) -> x0, x1; episode eligible[(x0 * n_elig) >> 32] over the held episodes
    with total >= length + 1 rows; start (x1 * (total - length + 1)) >> 32, or with balance
    min((x1 * total) >> 32, total - length)."""
    held = np.asarray(held, np.int64).reshape(-1, 2)
    elig = held[held[:, 1] >= length + 1]
    ids = np.full(batch, -1, np.int64)
    starts = np.full(batch, -1, np.int32)
    if len(elig) == 0:
        return ids, starts
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    x0, x1, _, _ = philox4x32_10(np.arange(batch), call, 0, 0, seed & 0xFFFFFFFF, (seed >> 32) ^ STREAM_STORE)
    pick = (x0.astype(np.uint64) * np.uint64(len(elig))) >> np.uint64(32)
    ids = elig[pick.astype(np.int64), 0]
    total = elig[pick.astype(np.int64), 1].astype(np.uint64)
    L = np.uint64(length)
    if balance:
        starts = np.minimum((x1.astype(np.uint64) * total) >> np.uint64(32), total - L)
    else:
        starts = (x1.astype(np.uint64) * (total - L + np.uint64(1))) >> np.uint64(32)
    return ids, starts.astype(np.int32)


# Random123 kat_vectors, philox4x32 with 10 rounds: (counter, key) -> output
KAT = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
       ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
        (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(ctr, key, want):
    got = philox4x32_10(*[np.array([v]) for v in ctr], *key)
    assert tuple(int(g[0]) for g in got) == want


def test_philox_equals_the_oracle(tmp_path):
    src = (ROOT / "oracle" / "rd_oracle.c").read_text()
    m = re.search(r"static void philox4x32_10\(.*?\n}\n", src, flags=re.S)
    assert m, "philox4x32_10 not found in oracle/rd_oracle.c"
    (tmp_path / "philox.c").write_text("#include <stdint.h>\n" + m.group(0) +
                                       "void philox_export(uint32_t* c, uint32_t k0, uint32_t k1) { philox4x32_10(c, k0, k1); }\n")
    so = tmp_path / "libphilox.so"
    subprocess.run(["cc", "-O2", "-shared", "-fPIC", "-o", str(so), str(tmp_path / "philox.c")], check=True)
    lib = C.CDLL(str(so))
    lib.philox_export.argtypes = [C.POINTER(C.c_uint32), C.c_uint32, C.c_uint32]
    rng = np.random.RandomState(3)
    ctr = rng.randint(0, 2 ** 32, size=(64, 4), dtype=np.uint64)
    keys = rng.randint(0, 2 ** 32, size=(64, 2), dtype=np.uint64)
    for c, k in zip(ctr, keys):
        buf = (C.c_uint32 * 4)(*[int(v) for v in c])
        lib.philox_export(buf, int(k[0]), int(k[1]))
        got = philox4x32_10(*[np.array([v]) for v in c], int(k[0]), int(k[1]))
        assert [int(g[0]) for g in got] == list(buf)


def test_draw_is_uniform_over_the_eligible_episodes():
    # 9 held episodes, 3 too short for L = 10 (they need 11 rows); 6 eligible
    held = [(0, 30), (1, 10), (2, 11), (3, 50), (4, 5), (5, 12), (6, 11), (7, 200), (8, 3)]
    ids = np.concatenate([store_draw(1234, k, 4096, 10, held)[0] for k in range(8)])
    eligible = [i for i, n in held if n >= 11]
    assert set(np.unique(ids)) == set(eligible)
    counts = np.array([(ids == i).sum() for i in eligible])
    assert stats.chisquare(counts).pvalue > 1e-3


@pytest.mark.parametrize("balance", [False, True])
def test_start_law(balance):
    total, L = 20, 5
    starts = np.concatenate([store_draw(99, k, 8192, L, [(7, total)], balance=balance)[1] for k in range(4)])
    assert starts.min() >= 0 and starts.max() <= total - L
    if balance:   # min(randint(0, total), total - L): the last start takes the mass of L values
        p = np.full(total - L + 1, 1.0 / total)
        p[-1] = L / total
    else:         # randint(0, total - L + 1)
        p = np.full(total - L + 1, 1.0 / (total - L + 1))
    counts = np.bincount(starts, minlength=total - L + 1)
    assert stats.chisquare(counts, p * len(starts)).pvalue > 1e-3


def test_draw_without_eligible_episodes():
    ids, starts = store_draw(0, 0, 16, 50, [(0, 10), (1, 50)])
    assert (ids == -1).all() and (starts == -1).all()


def test_draws_depend_on_seed_and_call():
    held = [(i, 100) for i in range(1000)]
    a = store_draw(5, 0, 64, 20, held)
    assert not np.array_equal(a[0], store_draw(5, 1, 64, 20, held)[0])
    assert not np.array_equal(a[0], store_draw(6, 0, 64, 20, held)[0])
    assert np.array_equal(a[0], store_draw(5, 0, 64, 20, held)[0])


def _cfg(**kw):
    cfg = _abi.RdConfig()
    cfg.action_repeat, cfg.dt, cfg.time_limit, cfg.task, cfg.agents_per_world = 4, 0.01, 180.0, _abi.TASK_MAX_PROGRESS, 1
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


def test_capacity_bound():
    # the task's time limit: done at the first tick with time > 180 s, tick 18001 at the latest -> 4501 steps of R 4
    assert max_episode_steps(_cfg()) == 4501
    assert max_episode_steps(_cfg(time_limit_steps=100)) == 100
    assert max_episode_steps(_cfg(time_limit_steps=10000)) == 4501
    assert max_episode_steps(_cfg(time_limit_ticks=10, action_repeat=4)) == 3
    assert max_episode_steps(_cfg(time_limit_ticks=12, action_repeat=4)) == 3
    assert max_episode_steps(_cfg(time_limit=1.0, action_repeat=8)) == 13     # ceil(102 / 8)
    # max_speed has no time limit: only the TimeLimit wrappers bound it
    assert max_episode_steps(_cfg(task=_abi.TASK_MAX_SPEED)) is None
    assert max_episode_steps(_cfg(task=_abi.TASK_MAX_SPEED, time_limit_ticks=400)) == 100
    # a world ends with its first car: one timed agent bounds it
    cfg = _cfg(agents_per_world=2)
    cfg.agent_task[0], cfg.agent_task[1] = _abi.TASK_MAX_SPEED, _abi.TASK_MAX_PROGRESS
    assert max_episode_steps(cfg) == 4501
    cfg.agent_task[1] = _abi.TASK_MAX_SPEED
    assert max_episode_steps(cfg) is None
