"""Import arena of the device-resident episode store on one GPU: what importing episodes costs and whether sampling over
imported episodes costs more than over recorded ones.  Prints (and with --out writes) one JSON object.

* insert() of the episodes a config-2 store recorded (follow-the-gap, 4096 envs), as float32 dicts, in GB/s of store
  rows written, against a plain pinned host -> device copy of the same bytes measured in the same run; and of some of
  them as float64 (converted on the device)
* load() of a directory of those episodes (np.savez_compressed files), decode included, against decoding the same
  files sequentially on the host alone
* sample(B = 50, L = 50) from a recorded-only, an imported-only and a mixed store holding the same episodes (recorded,
  imported, and both), alternated: tools/store_bench.py's
  CUDA-graph timing of the gather, draw + gather, and draw + gather with the eligibility compaction redone every call
  (the compaction then covers the recorded table and the arena's table)
* the card's name and power limit, read in the same run

    python tools/store_import_bench.py [--envs 4096] [--steps 253] [--files 200] [--out store_import_bench.json]
"""
import argparse
import json
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from store_bench import card, config, sample_throughput, timed  # noqa: E402

def row_bytes(store):
    return sum(int(np.prod(store._spec[k][0] or (1,))) * store._spec[k][1].itemsize for k in store.keys)


def make_store(torch, n, cap, import_rows, record_steps):
    from racing_dreamer_b200 import BatchedRaceEnv, GapFollowerPolicy
    from racing_dreamer_b200.episodes import DeviceEpisodeStore
    env = BatchedRaceEnv(config(("austria",), n, auto_reset=False), device="cuda:0")
    store = DeviceEpisodeStore(env, capacity_rows=cap, import_capacity_rows=import_rows, seed=3)
    if record_steps:
        store.reset()
        GapFollowerPolicy(env).rollout(record_steps, store=store)
    torch.cuda.synchronize()
    return store


def insert_rate(torch, store, eps, reps):
    rows = sum(len(e["reward"]) for e in eps)
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        store.insert(eps)
        torch.cuda.synchronize()
        out.append(time.perf_counter() - t0)
    written = rows * row_bytes(store)
    staged = sum(v.nbytes for ep in eps for v in ep.values())
    best = min(out)
    return {"episodes": len(eps), "rows": rows, "staged_bytes": staged, "written_bytes": written,
            "seconds": [round(t, 4) for t in out], "written_GB_per_s": round(written / best / 1e9, 2),
            "staged_GB_per_s": round(staged / best / 1e9, 2)}


def h2d_rate(torch, nbytes, reps):
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dev = torch.empty(nbytes, dtype=torch.uint8, device="cuda:0")
    dev.copy_(host, non_blocking=True)
    ms = [timed(torch, lambda: dev.copy_(host, non_blocking=True)) for _ in range(reps)]
    return {"bytes": nbytes, "ms": [round(m, 3) for m in ms], "GB_per_s": round(nbytes / min(ms) / 1e6, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=253)
    ap.add_argument("--files", type=int, default=200)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("store_import_bench.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    from racing_dreamer_b200.episodes import DeviceEpisodeStore, episode_files, save_episodes
    res = {"card": card(), "envs": a.envs, "record_steps": a.steps}
    cap = 2000 // 8 + 6
    # 253 recorded steps: nearly every env holds one whole episode of up to 251 rows, so the stores' episodes (GBs) do
    # not fit the L2 and the three stores below sample the same episodes: recorded, imported, and both
    recorded = make_store(torch, a.envs, cap, 0, a.steps)
    eps = recorded.episodes()
    rows = sum(len(e["reward"]) for e in eps)
    mixed = make_store(torch, a.envs, cap, rows, a.steps)
    imported = make_store(torch, a.envs, cap, rows, 0)
    res.update(row_bytes=row_bytes(mixed), episodes=len(eps), rows=rows, import_capacity_rows=rows)
    res["insert_float32"] = insert_rate(torch, imported, eps, a.reps)
    res["pinned_h2d_same_bytes"] = h2d_rate(torch, res["insert_float32"]["staged_bytes"], 5)
    sub = [{k: v.astype(np.float64) for k, v in e.items()} for e in eps[:a.files * 2]]
    res["insert_float64"] = insert_rate(torch, mixed, sub, a.reps)
    del sub
    mixed.insert(eps)            # as many rows as the arena: only these are held afterwards

    with tempfile.TemporaryDirectory() as tmp:
        save_episodes(tmp, eps[:a.files])
        files = episode_files(tmp)
        file_bytes = sum(f.stat().st_size for f in files)
        t0 = time.perf_counter()
        raw = 0
        for f in files:
            with np.load(f) as z:
                raw += sum(z[k].nbytes for k in z.files)
        decode_s = time.perf_counter() - t0
        loads = []
        for _ in range(a.reps):   # a new store each time: the arena starts empty
            st = DeviceEpisodeStore(imported.env, capacity_rows=cap, import_capacity_rows=rows, seed=3)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ids = st.load(tmp)
            torch.cuda.synchronize()
            loads.append(time.perf_counter() - t0)
        lrows = int(st.info()["imported_rows"])
        res["load_directory"] = {"files": len(files), "imported": len(ids), "rows": lrows, "file_bytes": file_bytes,
                                 "decoded_bytes": raw, "seconds": [round(t, 4) for t in loads],
                                 "written_GB_per_s": round(lrows * row_bytes(st) / min(loads) / 1e9, 3),
                                 "files_per_s": round(len(files) / min(loads), 1),
                                 "host_decode_only_sequential_s": round(decode_s, 4)}
        del st
    imported = DeviceEpisodeStore(imported.env, capacity_rows=cap, import_capacity_rows=rows, seed=3)
    imported.insert(eps)
    del eps
    res["stores"] = {name: s.info() for name, s in (("recorded_only", recorded), ("imported_only", imported),
                                                     ("mixed", mixed))}
    runs = {name: [] for name in res["stores"]}
    for rep in range(a.reps + 1):
        for name, s in (("recorded_only", recorded), ("imported_only", imported), ("mixed", mixed)):
            r = sample_throughput(torch, s)
            if rep > 0:   # the first round warms every shape up
                runs[name].append(r)
    res["sample_B50_L50"] = {
        name: {k: [r[k] for r in rs] for k in ("gather_us", "draw_plus_gather_us", "draw_plus_gather_with_compaction_us",
                                               "gather_GB_per_s", "python_sample_call_us")}
        for name, rs in runs.items()}
    for s in (recorded, imported, mixed):
        s.env.close()
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
