"""Device-resident episode store on one GPU: what recording costs in the closed loop, what sampling costs, and the host
path it replaces.  Prints (and with --out writes) one JSON object.

* closed loop, config 2 (austria, 4096 envs, action_repeat 8, random resets, 250-step time limit): follow-the-gap and
  the shipped Dreamer agent, un-recorded (today's rollout on an auto-resetting env) and recorded
  (``rollout(n, store=...)``), alternated in the same process; CUDA events around each rollout
* the same with obs_type='lidar_occupancy' on columbia (follow-the-gap)
* per-kernel device time of a recorded step and of sampling, from torch.profiler in a separate pass
* sample throughput at B = L = 50 (draws + gather; the eligibility list is cached while the store does not change) as
  bytes moved per second against the data sheet's 7.7 TB/s
* EpisodeRecorder over HostSteppedEnv on config 2 (numpy actions in, numpy episodes out)
* the card's name and power limit, read in the same run

    python tools/store_bench.py [--steps 200] [--reps 3] [--out store_bench.json]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

HBM_TBS = 7.7   # HGX B200 data sheet, one GPU


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def config(tracks, n, obs="lidar", auto_reset=True):
    from racing_dreamer_b200 import EnvConfig
    return EnvConfig(tracks=tracks, n_envs=n, action_repeat=8, obs_type=obs, auto_reset=auto_reset, reset_mode="random",
                     seed=1, time_limit_steps=2000 // 8)


def timed(torch, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def closed_loop(torch, tracks, n, obs, policies, steps, reps, capacity):
    from racing_dreamer_b200 import BatchedRaceEnv, DreamerPolicy, GapFollowerPolicy
    from racing_dreamer_b200.episodes import DeviceEpisodeStore
    arms = {}
    for rec in (False, True):
        env = BatchedRaceEnv(config(tracks, n, obs, auto_reset=not rec), device="cuda:0")
        store = DeviceEpisodeStore(env, capacity_rows=capacity) if rec else None
        pols = {}
        if "gap" in policies:
            pols["gap"] = GapFollowerPolicy(env)
        if "dreamer" in policies:
            pols["dreamer"] = DreamerPolicy(env, "austria_dreamer", noise="philox")
        if rec:
            store.reset()
        else:
            env.reset()
        arms[rec] = (env, store, pols)
    res = {}
    for name in policies:
        runs = {False: [], True: []}
        for rep in range(reps + 1):
            for rec in (False, True):
                env, store, pols = arms[rec]
                ms = timed(torch, lambda: pols[name].rollout(steps, store=store))
                if rep > 0:   # the first round warms every shape up
                    runs[rec].append(ms / steps)
        un, re = np.array(runs[False]), np.array(runs[True])
        res[name] = {"unrecorded_ms_per_step": un.round(4).tolist(), "recorded_ms_per_step": re.round(4).tolist(),
                     "unrecorded_Msteps_per_s": round(n / un.min() / 1e3, 2), "recorded_Msteps_per_s": round(n / re.min() / 1e3, 2),
                     "recording_overhead": round(float(np.median(re) / np.median(un) - 1.0), 4)}
    store = arms[True][1]
    info = store.info()
    for env, _, _ in arms.values():
        torch.cuda.synchronize()
    return res, info, arms


def kernel_profile(torch, env, store, pol, steps, n_samples):
    """Device time per kernel name over `steps` recorded steps and `n_samples` B = L = 50 draws (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    pol.rollout(2, store=store)
    store.sample(batch=50, length=50)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pol.rollout(steps, store=store)
        store.sample(batch=50, length=50)   # first draw after the store changed: eligibility compaction
        for _ in range(n_samples - 1):
            store.sample(batch=50, length=50)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0 or ev.count == 0:
            continue
        name = ev.key
        short = name.split("(")[0].split("<")[0]
        if "DeviceSelect" in name or "DeviceCompact" in name:
            short = "cub_select(" + ("init" if "Init" in name else "sweep") + ")"
        d = out.setdefault(short, {"calls": 0, "total_us": 0.0})
        d["calls"] += ev.count
        d["total_us"] += t
    for d in out.values():
        d["us_per_call"] = round(d["total_us"] / d["calls"], 2)
        d["total_us"] = round(d["total_us"], 1)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["total_us"]))


def sample_throughput(torch, store, reps=200):
    """B = L = 50.  Device time per launch from CUDA events around the replay of a CUDA graph of `reps` rd_store_sample
    calls (outputs preallocated, so neither the host nor launch gaps are in it): explicit indices = k_store_gather
    alone; drawing = k_store_draw + k_store_gather (eligibility list cached); drawing with the length alternating
    between 50 and 49 = + the cub compaction of the table window every call.  Python sample() calls (tensor
    allocation, ctypes, launch) are timed separately."""
    import ctypes as C
    env = store.env
    B = L = 50
    row = sum(int(np.prod(store._spec[k][0] or (1,))) * store._spec[k][1].itemsize for k in store.keys)
    moved = 2 * B * L * row      # every row read once from the rings and written once
    got = store.sample(batch=B, length=L)
    ids, starts = got["episode_id"].clone(), got["start"].clone()
    out = store.sample(length=L, indices=(ids, starts))
    b = store._abi.RdStoreBatch()
    for k, f in (("lidar", "lidar_dev"), ("lidar_occupancy", "occupancy_dev"), ("pose", "pose_dev"),
                 ("velocity", "velocity_dev"), ("speed", "speed_dev"), ("action", "action_dev"), ("reward", "reward_dev"),
                 ("discount", "discount_dev"), ("progress", "progress_dev"), ("time", "time_dev"),
                 ("episode_id", "episode_id_dev"), ("start", "start_dev")):
        if k in out:
            setattr(b, f, out[k].data_ptr())

    def call(explicit, length=L):
        env._check(env.lib.rd_store_sample(env._handle, B, length, 0, ids.data_ptr() if explicit else None,
                                            starts.data_ptr() if explicit else None, C.byref(b), env._stream()))

    def graph_ms(fn):
        fn(0)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for r in range(reps):
                fn(r)
        g.replay()
        torch.cuda.synchronize()
        return min(timed(torch, g.replay) for _ in range(5)) / reps

    gather_ms = graph_ms(lambda r: call(True))
    draw_ms = graph_ms(lambda r: call(False))
    compact_ms = graph_ms(lambda r: call(False, L - (r & 1)))
    store.sample(batch=B, length=L)
    py_ms = timed(torch, lambda: [store.sample(batch=B, length=L) for _ in range(reps)]) / reps
    gbs = moved / gather_ms / 1e6
    return {"batch": B, "length": L, "row_bytes": row, "bytes_per_sample": moved,
            "gather_us": round(gather_ms * 1e3, 2), "gather_GB_per_s": round(gbs, 1),
            "gather_fraction_of_7.7TB_s": round(gbs / (HBM_TBS * 1e3), 4),
            "draw_plus_gather_us": round(draw_ms * 1e3, 2),
            "draw_plus_gather_with_compaction_us": round(compact_ms * 1e3, 2),
            "table_slots": int(store.env.n * (store.capacity_rows + 2)),
            "python_sample_call_us": round(py_ms * 1e3, 2)}


def host_path(n, steps):
    from racing_dreamer_b200.episodes import EpisodeRecorder, max_episode_steps
    from racing_dreamer_b200.host import HostSteppedEnv
    env = HostSteppedEnv(config(("austria",), n, auto_reset=False), device="cuda:0", n_shards=8)
    eps = [0]
    rec = EpisodeRecorder(env, max_len=max_episode_steps(env.env.cfg), callbacks=[lambda e: eps.__setitem__(0, eps[0] + len(e))],
                          reset_mode="random")
    rec.reset()
    rng = np.random.RandomState(0)
    acts = rng.uniform(-1, 1, (8, n, 2)).astype(np.float32)
    acts[..., 0] = 0.6
    for t in range(3):
        rec.step(acts[t % 8])
    t0 = time.perf_counter()
    for t in range(steps):
        rec.step(acts[t % 8])
    dt = time.perf_counter() - t0
    env.close()
    return {"steps": steps, "ms_per_step": round(dt / steps * 1e3, 3), "Msteps_per_s": round(n * steps / dt / 1e6, 3),
            "episodes_committed": eps[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--host-steps", type=int, default=40)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("store_bench.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    n = a.envs
    res = {"card": card(), "envs": n, "steps_per_rollout": a.steps, "reps": a.reps}
    cap = 2000 // 8 + 6
    res["config2_closed_loop"], res["config2_store_info"], arms = closed_loop(
        torch, ("austria",), n, "lidar", ("gap", "dreamer"), a.steps, a.reps, cap)
    env, store, pols = arms[True]
    res["sample_B50_L50"] = sample_throughput(torch, store)
    res["kernels_recorded_gap_step_and_samples"] = kernel_profile(torch, env, store, pols["gap"], 20, 50)
    res["store_bytes"] = int(n * cap * sum(int(np.prod(store._spec[k][0] or (1,))) * store._spec[k][1].itemsize for k in store.keys))
    for e, _, _ in arms.values():
        e.close()
    del arms, env, store, pols
    torch.cuda.empty_cache()
    res["columbia_occupancy_closed_loop"], _, arms = closed_loop(
        torch, ("columbia",), n, "lidar_occupancy", ("gap",), max(20, a.steps // 4), a.reps, cap)
    for e, _, _ in arms.values():
        e.close()
    del arms
    torch.cuda.empty_cache()
    res["host_path_episode_recorder"] = host_path(n, a.host_steps)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
