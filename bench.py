#!/usr/bin/env python
"""bench.py -- env-steps/s (and LiDAR beams/s) of the batched racing-environment step on B200.

Contract (driver): `python bench.py --gpus N --steps K --warmup W [--impl reference]`; for N > 1 it is launched
under torchrun, one rank per GPU.  Rank 0 prints ONE JSON line.

Headline workload (BASELINE.json configs[1], SURVEY.md §8-d config 2): Austria track, 1080-beam LiDAR, 4096 batched
envs per GPU, action_repeat 8, obs 'lidar' f32, reset mode 'random' (seed 1), scripted actions motor=+0.6,
steering=0.8*sin(2*pi*k/50 + phi_i), auto-reset on.  A "step" = one BatchedRaceEnv.step() -- the public API -- of the
whole batch.

* value       device-resident env-steps/s: actions already in HBM, outputs stay in HBM; CUDA events per step
              on the launching stream, L2 flushed between steps (outside the events); max over ranks.
* e2e         the same metric through the host-facing call (HostSteppedEnv.step: numpy actions in pinned
              memory -> H2D -> kernels -> D2H of every observation/result array -> numpy), wall clock.
              Siblings (top level): e2e_f16 (scans stored as IEEE half = Collect at precision 16) and
              e2e_two_groups_async (two half-batches through step_async / step_wait).
* roofline    the dominant kernel of the step: algorithmic bytes per launch / its mean launch duration (CUDA events
              inside librd_env, rd_enable_timing), against MEASURED_PEAKS.json hbm_gbs.
* configs     the other BASELINE configs (3: Columbia lidar_occupancy 16384 envs; 4: Treitlstrasse random actions 65536
              envs, terminations/s; 5: Barcelona+Austria 131072 envs per GPU) as short legs of the same run, each with
              value / kernel_ms / roofline / e2e, so that the driver's BENCH and SCALE files carry all of them.
* cpu_baseline  the CPU oracle (oracle/rd_oracle.c, kind "port") on all host threads, bounded sample, on rank 0 at every
              N; plus `reference_stack`: BASELINE config 1 -- the reference's UNMODIFIED wrapper stack over the one-tick
              oracle env, 1 env, 1 core (live when /root/reference exists, else the committed measurement).
* --impl reference  the reference arm: the same oracle port timed on the host cores (the reference's env
              arithmetic lives in un-vendored racecar_gym + pybullet, so no reference build exists: DESIGN.md).
* --dump-outputs DIR  what the headline's last timed step returned (obs, reward, done, info) as DIR/<name>.npy in
              float32 / float64, at most 64 MB (beyond that a fixed sample of envs).  The inputs depend only on the
              arguments, so the files of two builds can be compared array by array.
"""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_BEAMS = 1080
ACTION_REPEAT = 8
PERIOD = 50
# BASELINE.json configs[1..4] (SURVEY.md §8-d).  The driver's bench line is config 2; the others are legs of the same run
# (`--config N` makes any of them the headline instead).
CONFIGS = {
    2: dict(tracks=("austria",), envs=4096, obs="lidar", actions="scripted", seed=1),
    3: dict(tracks=("columbia",), envs=16384, obs="lidar_occupancy", actions="scripted", seed=3),
    4: dict(tracks=("treitlstrasse_v2",), envs=65536, obs="lidar", actions="random", seed=4),
    5: dict(tracks=("barcelona", "austria"), envs=131072, obs="lidar", actions="scripted", seed=5),
}
# SURVEY.md §8-d: state r/w 224 + action 8 + lidar 4320 + scalars 24 + pose/velocity 48
ALGO_BYTES_PER_ENV_STEP = 4624
# per kernel: k_lidar writes 1080 f32 ranges and reads one 48-byte origin record per env; k_occupancy writes 64x64 u8 and
# reads the record + pose; k_step reads and writes the state groups, reads the action, writes scalars + pose/velocity + record
KERNEL_BYTES_PER_ENV = {"k_lidar": N_BEAMS * 4 + 48, "k_occupancy": 4096 + 48 + 24, "k_step": 224 + 8 + 24 + 48 + 48}
# --dump-outputs: total size of the .npy files written
DUMP_LIMIT_BYTES = 64 * 10**6


@dataclasses.dataclass
class Workload:
    cfg_id: int
    tracks: tuple
    envs: int
    obs: str
    actions: str
    seed: int

    def name(self):
        return (f"config{self.cfg_id}: {'+'.join(self.tracks)} {N_BEAMS}-beam lidar, {self.envs} envs/GPU, "
                f"action_repeat={ACTION_REPEAT}, obs={self.obs}, {self.actions} actions")


def workload_of(cfg_id, envs=0, obs=""):
    c = CONFIGS[cfg_id]
    return Workload(cfg_id, c["tracks"], envs or c["envs"], obs or c["obs"], c["actions"], c["seed"])


def scripted_actions(wl, n, rank=0):
    """[PERIOD, n, 2] float32: motor +0.6, steering 0.8*sin(2*pi*k/50 + phi_i), phi_i from a seeded stream
    (config 4: uniform random U(-1,1)^2 instead, so that collisions / laps / time limits fire)."""
    rng = np.random.Generator(np.random.Philox(key=2 + 1000 * rank))
    if wl.actions == "random":
        return rng.uniform(-1.0, 1.0, (PERIOD, n, 2)).astype(np.float32)
    phi = rng.uniform(0.0, 2.0 * np.pi, n)
    k = np.arange(PERIOD)[:, None]
    a = np.empty((PERIOD, n, 2), np.float32)
    a[..., 0] = 0.6
    a[..., 1] = (0.8 * np.sin(2.0 * np.pi * k / PERIOD + phi[None, :])).astype(np.float32)
    return a


def env_config(wl, n_envs, rank=0, **over):
    from racing_dreamer_b200 import EnvConfig
    kw = dict(tracks=wl.tracks, n_envs=n_envs, action_repeat=ACTION_REPEAT, obs_type=wl.obs, auto_reset=True,
              reset_mode="random", seed=wl.seed, env_id_offset=rank * n_envs, time_limit_steps=2000 // ACTION_REPEAT)
    kw.update(over)
    return EnvConfig(**kw)


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", d
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)", {}


def ncu_entry(config_id, n_envs, kernel):
    """The committed ncu capture of `kernel` for this workload (profiles/ncu_traffic.json), or None."""
    try:
        ent = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text()).get(f"config{config_id}", {}).get(kernel)
        if ent and int(ent["envs"]) == int(n_envs):
            return ent
    except (OSError, ValueError, KeyError):
        pass
    return None


def ncu_on_chip(config_id, n_envs, kernel, sm_count=148):
    """The on-chip picture of `kernel` from the committed ncu capture (SURVEY.md §8-d asks for both): issue-slot
    utilisation and the share of the shared-memory pipe its wavefronts use; None without a matching capture."""
    ent = ncu_entry(config_id, n_envs, kernel)
    if not ent or "issue_active_pct" not in ent:
        return None
    out = {"bound": "issue slots", "issue_active_pct": ent["issue_active_pct"],
           "smem_pipe_frac": ent["smem_wavefronts"] / (sm_count * ent["sm_cycles_elapsed"]),
           "source": ent["source"] + " (ncu --set full, one launch)"}
    if "active_lanes_per_inst" in ent:
        out["active_lanes_per_warp_inst"] = ent["active_lanes_per_inst"]
    if kernel == "k_lidar" and "warp_inst_executed" in ent:
        out["warp_inst_per_beam_group"] = ent["warp_inst_executed"] / (n_envs * ((N_BEAMS + 31) // 32))
    if "bank_conflict_wavefronts" in ent:
        out["smem_bank_conflict_frac"] = ent["bank_conflict_wavefronts"] / max(1, ent["smem_wavefronts"])
    return out


def ncu_traffic(config_id, n_envs, kernel):
    ent = ncu_entry(config_id, n_envs, kernel)
    return None if not ent else int(ent["dram_read_bytes"]) + int(ent["dram_write_bytes"])


def roofline_of(wl, n, timing, step_ms_total, value_per_gpu):
    """`roofline` object for the kernel that takes most of the step."""
    per = {"k_step": timing["step_ms"] / max(1, timing["step_launches"]),
           "k_lidar": timing["lidar_ms"] / max(1, timing["lidar_launches"]),
           "k_occupancy": timing["occupancy_ms"] / max(1, timing["occupancy_launches"])}
    tot = {"k_step": timing["step_ms"], "k_lidar": timing["lidar_ms"], "k_occupancy": timing["occupancy_ms"]}
    kern = max(tot, key=tot.get)
    launches = {"k_step": timing["step_launches"], "k_lidar": timing["lidar_launches"], "k_occupancy": timing["occupancy_launches"]}[kern]
    # a launch of k_lidar / k_occupancy handles the envs of ONE track (envs alternate between the tracks).  With several
    # tracks only the first track's launch is event-bracketed: the others run on streams of their own and queue behind
    # its persistent CTAs, so `per` is that launch's time and the bytes are that launch's.
    envs_per_launch = n / len(wl.tracks) if kern != "k_step" else n
    algo = KERNEL_BYTES_PER_ENV[kern] * envs_per_launch
    peak, peak_src, _ = measured_peaks()
    gbs = algo / (per[kern] * 1e-3) / 1e9 if per[kern] > 0 else 0.0
    return per, {"bound": "hbm", "kernel": kern, "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                 "traffic": ncu_traffic(wl.cfg_id, n, kern), "peak_source": peak_src, "kernel_ms": per[kern],
                 "kernel_share_of_step": tot[kern] / max(step_ms_total, 1e-9),
                 "algorithmic_bytes_per_launch": algo,
                 "step_algorithmic_gbs": (ALGO_BYTES_PER_ENV_STEP + (4096 if wl.obs == "lidar_occupancy" else 0)) * value_per_gpu / 1e9,
                 "on_chip": ncu_on_chip(wl.cfg_id, n, kern),
                 "note": "on-chip bound (instruction issue / shared memory; the map lives in shared memory), see DESIGN.md"}


# --------------------------------------------------------------------------------------------- CPU arms
def cpu_oracle_run(wl, n_envs, steps, warmup, threads, rank=0):
    """Times the oracle port on `threads` host threads: `steps` env.step() calls of `n_envs` envs."""
    from oracle import Oracle, default_config
    from racing_dreamer_b200 import _abi, load_track
    from racing_dreamer_b200.env import _fill_config
    cfg = default_config()
    _fill_config(cfg, env_config(wl, n_envs, rank))
    ids = (np.arange(n_envs) % len(wl.tracks)).astype(np.int32)
    orc = Oracle(cfg, [load_track(t) for t in wl.tracks], ids, n_threads=threads)
    orc.reset(mode=_abi.RESET_RANDOM)
    acts = scripted_actions(wl, n_envs, rank)
    for k in range(warmup):
        orc.step(acts[k % PERIOD])
    t0 = time.perf_counter()
    for k in range(steps):
        orc.step(acts[(warmup + k) % PERIOD])
    dt = time.perf_counter() - t0
    return n_envs * steps / dt, dt


def cpu_baseline_of(wl, budget_s=1.5):
    threads = os.cpu_count() or 1
    rate, _ = cpu_oracle_run(wl, 256 if wl.obs == "lidar" else 2 * threads, 2, 1, threads)
    n_s = int(min(wl.envs, max(threads, rate * 1.0)))          # <= ~1 s per step
    steps_s = int(min(200, max(12 if wl.obs == "lidar" else 3, budget_s * rate / n_s)))
    v, dt = cpu_oracle_run(wl, n_s, steps_s, 1, threads)
    return {"value": v, "unit": "env-steps/s", "cores": threads, "kind": "port",
            "sample": f"{n_s} envs x {steps_s} steps of the same workload, oracle/rd_oracle.c, {threads} OpenMP threads, {dt:.1f} s"}


def reference_stack_baseline(steps=1000):
    """BASELINE config 1 / BASELINE.md C1: the reference's UNMODIFIED wrapper stack [REF dreamer/dream.py:103-140;
    dreamer/wrappers.py:22-250] over the one-tick oracle env: 1 env, Columbia, obs lidar_occupancy (dream.py's stack always
    carries OccupancyMapObs), action_repeat 4, random actions, 1 core.  Needs /root/reference (the wrappers are imported
    from there, nothing is copied); on a box without it the committed measurement is reported instead."""
    committed = None
    try:
        committed = json.loads((ROOT / "profiles" / "r2_reference_stack_cpu.json").read_text())
    except (OSError, ValueError):
        pass
    try:
        from oracle import ref_stubs
        if not ref_stubs.available():
            raise RuntimeError("no /root/reference on this host")
        from oracle.ref_env import make_reference_stack
        from racing_dreamer_b200 import load_track
        env = make_reference_stack(load_track("columbia"), action_repeat=4, time_limit_steps=500, reset_mode="grid")
        acts = np.random.RandomState(0).uniform(-1, 1, (steps, 2)).astype(np.float32)
        env.reset()
        t0 = time.perf_counter()
        for k in range(steps):
            _, _, dones, _ = env.step({"A": acts[k]})
            if dones["A"]:
                env.reset()
        dt = time.perf_counter() - t0
        return {"value": steps / dt, "unit": "env-steps/s", "cores": 1,
                "kind": "reference wrapper stack (unmodified) over the oracle's one-tick env",
                "sample": f"1 env x {steps} agent steps, columbia, action_repeat 4, lidar_occupancy, random actions, {dt:.1f} s",
                "where": "live (this host)", "sim_ticks_per_s": 4 * steps / dt}
    except Exception as e:  # noqa: BLE001 -- the GPU box has no reference tree
        if committed:
            committed = dict(committed)
            committed["where"] = f"committed measurement (profiles/r2_reference_stack_cpu.json, build container): {e}"
            return committed
        return {"unavailable": str(e)}


def reference_arm(args, wl):
    """`--impl reference`: the reference's CPU env path on the host cores.  The reference is Python whose env
    arithmetic lives in un-vendored racecar_gym + pybullet (not installable offline), so this times the oracle
    port (oracle/rd_oracle.c) with every host thread, on the same config/metric as our arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    # size each step (env sample) so that steps+warmup finish in about two minutes
    rate, _ = cpu_oracle_run(wl, 256, 2, 1, threads)
    total_steps = max(1, args.steps + args.warmup)
    n_sample = int(min(wl.envs, max(threads, rate * 110.0 / total_steps)))
    value, dt = cpu_oracle_run(wl, n_sample, args.steps, args.warmup, threads)
    line = {
        "metric": "env_steps_per_s", "value": value, "unit": "env-steps/s", "impl": "reference", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "beams_per_s": value * N_BEAMS,
        "config": {"workload": wl.name(), "sample": f"{n_sample} of {wl.envs} envs per step"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{n_sample} envs x {args.steps} steps, oracle/rd_oracle.c, {threads} OpenMP threads",
                         "reference_stack": reference_stack_baseline(300)},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------------------------- GPU legs
class Ctx:
    """torch / distributed plumbing shared by the legs."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device(f"cuda:{self.local}")
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)   # > 126 MB L2

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def sum_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in t]


def step_outputs(obs, reward, done, info, limit=DUMP_LIMIT_BYTES):
    """What one BatchedRaceEnv.step() handed its caller, as host arrays with one row per env: floats as they are, other
    types converted exactly (to float32 up to two bytes, else float64).  When the rows exceed `limit` bytes, a fixed
    sample of envs (seed 0, ascending) is taken from every array alike and its indices are added as `env_index`."""
    import torch
    named = {}
    for k, v in list(obs.items()) + [("reward", reward), ("done", done)] + list(info.items()):
        named.setdefault(k, v)

    def host_dtype(t):
        if t.dtype in (torch.float32, torch.float64):
            return t.dtype
        return torch.float32 if t.element_size() <= 2 else torch.float64

    n = reward.shape[0]
    per_env = sum(t[0].numel() * torch.empty((), dtype=host_dtype(t)).element_size() for t in named.values())
    m = min(n, (limit - 4096) // (per_env + 8))      # 4 KiB for the .npy headers, 8 bytes per env for env_index
    rows = None
    if m < n:
        rows = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, m, replace=False))).to(reward.device)
    out = {}
    for k, t in named.items():
        if rows is not None:
            t = t.index_select(0, rows)
        out[k] = t.to(host_dtype(t)).cpu().numpy()
    if rows is not None:
        out["env_index"] = rows.cpu().numpy().astype(np.float64)
    return out


def device_leg(cx, wl, n, steps, warmup, sampler=None, back_to_back=True, keep_outputs=False):
    """K steps of BatchedRaceEnv.step() with inputs resident in HBM; per-step CUDA events, L2 flushed between steps.
    keep_outputs: also return what the last timed step returned (`step_outputs`), copied after the timed region."""
    torch = cx.torch
    from racing_dreamer_b200 import BatchedRaceEnv
    env = BatchedRaceEnv(env_config(wl, n, cx.rank), device=cx.dev)
    acts = torch.from_numpy(scripted_actions(wl, n, cx.rank)).to(cx.dev)      # inputs resident in HBM before timing
    env.reset()
    for k in range(warmup):
        env.step(acts[k % PERIOD])
    env.read_stats(reset=True)
    cx.barrier()
    if sampler:
        sampler.start()
    env.enable_timing(True)
    env.read_timing(reset=True)
    launches0 = env.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    cx.barrier()
    wall0 = time.perf_counter()
    for k in range(steps):
        cx.flush.zero_()
        ev[k][0].record()
        last = env.step(acts[(warmup + k) % PERIOD])      # the public API (launches only k_* kernels)
        ev[k][1].record()
    cx.barrier()
    wall = time.perf_counter() - wall0
    launches = env.launch_count - launches0
    timing = env.read_timing(reset=True)
    env.enable_timing(False)
    outputs = step_outputs(*last) if keep_outputs else None
    gpu_ms = float(sum(a.elapsed_time(b) for a, b in ev))
    stats = env.read_stats()
    b2b_ms = 0.0
    if back_to_back:   # no flush, one event pair
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cx.barrier()
        b0.record()
        for k in range(steps):
            env.step(acts[k % PERIOD])
        b1.record()
        cx.barrier()
        b2b_ms = b0.elapsed_time(b1)
    clocks = sampler.stop() if sampler else None
    gpu_ms_max, b2b_ms_max = cx.max_over_ranks(gpu_ms, b2b_ms)
    env.close()
    value = cx.world * n * steps / (gpu_ms_max / 1e3)
    per, roof = roofline_of(wl, n, timing, gpu_ms, value / cx.world)
    return {"value": value, "ms_per_step": gpu_ms_max / steps,
            "ms_per_step_back_to_back": b2b_ms_max / steps if back_to_back else None,
            "kernel_ms": per, "roofline": roof, "launches": int(launches), "wall_s": wall, "stats": stats, "clocks": clocks,
            "steps": steps, "warmup": warmup, "outputs": outputs}


def e2e_leg(cx, wl, n, steps, shards, **over):
    """The host-facing call: numpy actions -> pinned -> H2D -> step -> D2H of all results -> numpy, wall clock."""
    from racing_dreamer_b200.host import HostSteppedEnv
    henv = HostSteppedEnv(env_config(wl, n, cx.rank, **over), device=cx.dev, n_shards=shards, bind_cpu=cx.world > 1)
    hacts = scripted_actions(wl, n, cx.rank)
    henv.reset()
    for k in range(3):
        henv.step(hacts[k % PERIOD])
    cx.barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        out = henv.step(hacts[(3 + k) % PERIOD])
    cx.torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    assert out["lidar"].shape == (n, N_BEAMS) and np.isfinite(out["reward"]).all()
    h2d, d2h, nsh = henv.h2d_bytes_per_step, henv.d2h_bytes_per_step, len(henv.shards)
    henv.close()
    (dt_max,) = cx.max_over_ranks(dt)
    return {"value": cx.world * n * steps / dt_max, "unit": "env-steps/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "steps": steps, "shards": nsh, "ms_per_step": dt_max / steps * 1e3}


def two_groups_leg(cx, wl, n, steps, shards):
    """The same call split in two (step_async / step_wait) over two half-batches: group A's kernels run while group B's
    results cross PCIe -- the asynchronous vector-env pattern."""
    from racing_dreamer_b200.host import HostSteppedEnv
    if n % 2:
        return None
    half = n // 2
    hacts = scripted_actions(wl, n, cx.rank)
    groups = [HostSteppedEnv(env_config(wl, half, cx.rank, env_id_offset=cx.rank * n + g * half), device=cx.dev,
                             n_shards=max(1, shards // 2), bind_cpu=cx.world > 1) for g in range(2)]
    for g in groups:
        g.reset()
    acts2 = [np.ascontiguousarray(hacts[:, :half]), np.ascontiguousarray(hacts[:, half:])]
    for k in range(3):
        for g in range(2):
            groups[g].step(acts2[g][k % PERIOD])
    cx.barrier()
    t0 = time.perf_counter()
    groups[0].step_async(acts2[0][3 % PERIOD])
    for k in range(steps):
        groups[1].step_async(acts2[1][(3 + k) % PERIOD])
        o0 = groups[0].step_wait()
        if k + 1 < steps:
            groups[0].step_async(acts2[0][(4 + k) % PERIOD])
        o1 = groups[1].step_wait()
    dt = time.perf_counter() - t0
    assert o0["lidar"].shape == (half, N_BEAMS) and np.isfinite(o1["reward"]).all()
    d2h = sum(g.d2h_bytes_per_step for g in groups)
    for g in groups:
        g.close()
    (dt_max,) = cx.max_over_ranks(dt)
    return {"value": cx.world * n * steps / dt_max, "unit": "env-steps/s", "ms_per_step": dt_max / steps * 1e3,
            "h2d_bytes_per_step": n * 8, "d2h_bytes_per_step": d2h, "steps": steps,
            "note": "two half-batches through step_async/step_wait (rd_step_host_begin/_end): one group's kernels overlap "
                    "the other's device->host copy; same bytes per env-step"}


def d2h_probe(cx, mb=64, reps=5):
    """Pinned device->host copy rate: this rank alone, and every rank at the same time (the host fabric's ceiling for the
    host-facing step at N GPUs)."""
    torch = cx.torch
    probe_d = torch.empty(mb << 20, dtype=torch.uint8, device=cx.dev)
    probe_h = torch.empty(mb << 20, dtype=torch.uint8, pin_memory=True)

    def run():
        probe_h.copy_(probe_d, non_blocking=True)
        torch.cuda.synchronize()
        tp = time.perf_counter()
        for _ in range(reps):
            probe_h.copy_(probe_d, non_blocking=True)
        torch.cuda.synchronize()
        return reps * (mb << 20) / (time.perf_counter() - tp) / 1e9

    alone = 0.0
    for r in range(cx.world):       # one rank at a time
        cx.barrier()
        if r == cx.rank:
            alone = run()
        cx.barrier()
    together = run()                 # all ranks concurrently
    cx.barrier()
    (agg,) = cx.sum_over_ranks(together)
    (neg_min,) = cx.max_over_ranks(-together)
    return alone, together, agg, -neg_min


def closed_loop_leg(cx, wl, n, steps, warmup):
    """An on-device policy drives every env, no host round trip per step (SURVEY §8-f2)."""
    torch = cx.torch
    from racing_dreamer_b200 import BatchedRaceEnv, DreamerPolicy, GapFollowerPolicy
    closed = {}
    _, _, peaks = measured_peaks()
    for pname in ("follow_the_gap", "dreamer"):
        cenv = BatchedRaceEnv(env_config(wl, n, cx.rank), device=cx.dev)
        pol = GapFollowerPolicy(cenv) if pname == "follow_the_gap" else DreamerPolicy(cenv, "austria_dreamer", noise="philox")
        cenv.reset()
        pol.rollout(warmup)
        cenv.read_stats(reset=True)
        cenv.enable_timing(True)
        cenv.read_timing(reset=True)
        l0 = cenv.launch_count
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cx.barrier()
        c0.record()
        pol.rollout(steps)
        c1.record()
        cx.barrier()
        (tc,) = cx.max_over_ranks(c0.elapsed_time(c1))
        ct = cenv.read_timing(reset=True)
        cstats = cenv.read_stats()
        policy_ms = ct["policy_ms"] / max(1, ct["policy_launches"])
        leg = {"value": cx.world * n * steps / (tc / 1e3), "unit": "env-steps/s", "steps": steps,
               "ms_per_step": tc / steps, "launches_per_step": (cenv.launch_count - l0) / steps,
               "kernel_ms": {"policy": policy_ms, "k_step": ct["step_ms"] / max(1, ct["step_launches"]),
                             "k_lidar": ct["lidar_ms"] / max(1, ct["lidar_launches"])},
               "episode_stats_rank0": cstats}
        if pname == "follow_the_gap":
            leg["policy"] = "follow_the_gap on device (k_gap_follower), back-to-back steps"
        else:
            # multiply-accumulates of one RacingDreamer.action: img1 + GRU + obs1 + obs2 + actor (h0..h3, hout)
            macs = 32 * 200 + 2 * 200 * 600 + 1280 * 200 + 200 * 60 + 230 * 400 + 3 * 400 * 400 + 400 * 4
            tf = 2.0 * macs * n / (policy_ms * 1e-3) / 1e12
            bf16 = float(peaks.get("bf16_tflops", 1590.0))
            leg["policy"] = ("shipped Dreamer agent austria_dreamer on device: k_embed_lidar + k_dense launches + k_dense_chain "
                             "(the actor trunk in one launch) + k_actor_mode (tcgen05 kind::tf32, hi/lo x3 products, "
                             "float32-grade), Philox draws, back-to-back steps")
            leg["roofline"] = {"bound": "tensor", "kernel": "k_dense", "achieved": tf, "unit": "TFLOP/s",
                               "executed_tf32_tflops": 3.0 * tf, "peak": bf16 / 2.0,
                               "peak_source": ("measured bf16 cuBLAS peak / 2 (TF32 runs at half the bf16 rate)" if peaks else
                                               "fallback 1.59 PFLOP/s bf16 / 2"),
                               "frac": 3.0 * tf / (bf16 / 2.0), "flops_per_env_step": 2 * macs,
                               "note": "latency-bound at this batch: eight dependent launches of 32-128 CTAs each"}
        closed[pname] = leg
        cenv.close()
    return closed


def multi_agent_leg(cx, wl, n, steps, warmup):
    """The same car count as worlds of four cars that see and hit each other, tasks of the baselines' scenario files
    (A maximize_progress, B..D n_step_progress), reset 'random_ball' (SURVEY §8-f3)."""
    torch = cx.torch
    from racing_dreamer_b200 import BatchedRaceEnv
    mec = env_config(wl, n, cx.rank, reset_mode="random_ball", agents_per_world=4,
                     agent_tasks=("maximize_progress",) + ("n_step_progress",) * 3)
    menv = BatchedRaceEnv(mec, device=cx.dev)
    acts = torch.from_numpy(scripted_actions(wl, n, cx.rank)).to(cx.dev)
    menv.reset()
    for k in range(warmup):
        menv.step(acts[k % PERIOD])
    menv.read_stats(reset=True)
    menv.enable_timing(True)
    menv.read_timing(reset=True)
    mev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    cx.barrier()
    for k in range(steps):
        cx.flush.zero_()
        mev[k][0].record()
        menv.step(acts[(warmup + k) % PERIOD])
        mev[k][1].record()
    cx.barrier()
    (tm_,) = cx.max_over_ranks(float(sum(a.elapsed_time(b) for a, b in mev)))
    mt = menv.read_timing(reset=True)
    mstats = menv.read_stats()
    contacts = int((menv.buf["opponents"] != 0).sum())
    menv.close()
    return {"value": cx.world * n * steps / (tm_ / 1e3), "unit": "env-steps/s (cars)", "steps": steps,
            "ms_per_step": tm_ / steps, "worlds_per_gpu": n // 4, "agents_per_world": 4,
            "kernel_ms": {"k_step_ma": mt["step_ms"] / max(1, mt["step_launches"]),
                          "k_lidar": mt["lidar_ms"] / max(1, mt["lidar_launches"]),
                          "k_occupancy": mt["occupancy_ms"] / max(1, mt["occupancy_launches"])},
            "cars_in_contact_last_step_rank0": contacts, "episode_stats_rank0": mstats,
            "note": "worlds of 4 cars (tasks A maximize_progress, B..D n_step_progress), scans see the other cars, "
                    "world-level ActionRepeat/TimeLimit/reset; L2 flushed between steps"}


def config_leg(cx, cfg_id, steps, e2e_steps, shards):
    """One of the other BASELINE configs as a short leg: device-resident value + per-kernel split + roofline + e2e."""
    wl = workload_of(cfg_id)
    n = wl.envs
    d = device_leg(cx, wl, n, steps, 3, back_to_back=False)
    e = e2e_leg(cx, wl, n, e2e_steps, shards)
    leg = {"workload": wl.name(), "value": d["value"], "unit": "env-steps/s", "beams_per_s": d["value"] * N_BEAMS,
           "n_gpus": cx.world, "steps": d["steps"], "warmup": d["warmup"], "ms_per_step": d["ms_per_step"],
           "kernel_ms": d["kernel_ms"], "roofline": d["roofline"], "gpu_launches": d["launches"], "e2e": e,
           "l2": "flushed between steps", "episode_stats_rank0": d["stats"]}
    if cfg_id == 4:   # collisions / laps / time limits fire: terminations per second of device time
        leg["terminations_per_s"] = cx.world * d["stats"]["episodes"] / (d["ms_per_step"] * d["steps"] / 1e3)
    if cfg_id == 5 and n % 8 == 0:
        # Strong scaling of this config needs no second box: the envs shard with no exchange, so the step time of an
        # 8-GPU job over these n envs IS one GPU's step time over n/8 envs (measured here, same flush, same events).
        s = device_leg(cx, wl, n // 8, steps, 3, back_to_back=False)
        leg["strong_shard_of_8"] = {"envs_per_gpu": n // 8, "ms_per_step": s["ms_per_step"], "kernel_ms": s["kernel_ms"],
                                    "speedup_over_one_gpu": d["ms_per_step"] / s["ms_per_step"],
                                    "note": "time of one of eight shards of the same batch; no collective in step"}
    return leg


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="headline BASELINE.json config (default 2)")
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU of the headline (0 = the config's)")
    ap.add_argument("--obs", default="", choices=["", "lidar", "lidar_occupancy"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-closed-loop", action="store_true", help="skip the on-device policy rollout leg")
    ap.add_argument("--no-multi-agent", action="store_true", help="skip the four-cars-per-world leg (SURVEY §8-f3)")
    ap.add_argument("--no-configs", action="store_true", help="skip the legs of the other BASELINE configs")
    ap.add_argument("--no-e2e-variants", action="store_true", help="skip e2e_f16 / e2e_two_groups_async")
    ap.add_argument("--config-steps", type=int, default=0, help="timed steps of the other configs' legs (0 = min(steps, 20))")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 200)")
    ap.add_argument("--e2e-shards", type=int, default=8, help="stream shards of the host-facing env")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned (rank 0's envs) as DIR/<name>.npy, float32/float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    wl = workload_of(args.config, args.envs, args.obs)
    if args.impl == "reference":
        return reference_arm(args, wl)

    # stdout carries exactly ONE JSON line: anything native libraries print on fd 1 meanwhile (NCCL's version banner
    # when NCCL_DEBUG is set on the box) goes to stderr instead.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    cx = Ctx()
    n = wl.envs
    main_leg = device_leg(cx, wl, n, args.steps, args.warmup, sampler=ClockSampler(cx.local) if cx.rank == 0 else None,
                          keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and cx.rank == 0:
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        for name, a in main_leg.pop("outputs").items():
            np.save(out_dir / f"{name}.npy", a)

    e2e_steps = args.e2e_steps or min(args.steps, 200)
    e2e = e2e_leg(cx, wl, n, e2e_steps, args.e2e_shards)
    alone, together, agg, mn = d2h_probe(cx)
    e2e["pinned_d2h_gbs"] = alone
    e2e["d2h_floor_ms"] = e2e["d2h_bytes_per_step"] / alone / 1e6
    if cx.world > 1:   # the host fabric shared by all ranks: what N concurrent plain copies reach in this very run
        e2e["pinned_d2h_gbs_all_ranks_concurrent"] = {"aggregate": agg, "min_rank": mn, "this_rank": together}
        e2e["d2h_floor_ms_concurrent"] = e2e["d2h_bytes_per_step"] / mn / 1e6
    e2e_f16 = two = None
    if not args.no_e2e_variants:
        if wl.obs == "lidar":
            e2e_f16 = e2e_leg(cx, wl, n, e2e_steps, args.e2e_shards, lidar_dtype="float16")
            e2e_f16["note"] = ("scans stored as IEEE half: what the reference's Collect hands on at precision 16 "
                               "[REF dreamer/wrappers.py:240-250; dreamer/dream.py:176-177]")
        two = two_groups_leg(cx, wl, n, e2e_steps, args.e2e_shards)
    e2e["two_groups_async"] = two

    closed = None if args.no_closed_loop else closed_loop_leg(cx, wl, n, min(args.steps, 500), args.warmup)
    multi = None if (args.no_multi_agent or n % 4) else multi_agent_leg(cx, wl, n, min(args.steps, 300), args.warmup)

    configs = None
    if not args.no_configs:
        cs = args.config_steps or min(args.steps, 20)
        configs = {}
        for cid in sorted(CONFIGS):
            if cid == args.config:
                continue
            configs[f"config{cid}"] = config_leg(cx, cid, cs, max(3, min(cs, 8)), args.e2e_shards)

    # ---- the only collective of the system: episode statistics gathered across ranks at log cadence ----
    from racing_dreamer_b200.stats import gather_stats
    stats_all, _ = gather_stats(main_leg["stats"], device=cx.dev)

    if cx.rank == 0:
        value = main_leg["value"]
        line = {
            "metric": "env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": cx.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main_leg["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64 dynamics / i32 ray march / f32 ranges", "data": "synthetic",
            "beams_per_s": value * N_BEAMS,
            "sim_ticks_per_s": value * ACTION_REPEAT,
            "config": {"workload": wl.name(), "envs_per_gpu": n, "api": "BatchedRaceEnv.step()",
                       "l2": "flushed between steps (256 MiB memset outside the per-step events)",
                       "parallelism": f"env-sharded x{cx.world}, no collective in step"},
            "ms_per_step_back_to_back": main_leg["ms_per_step_back_to_back"],
            "wall_s_timed_region": main_leg["wall_s"],
            "roofline": main_leg["roofline"],
            "kernel_ms": main_leg["kernel_ms"],
            "e2e": e2e,
            "e2e_f16": e2e_f16,
            "e2e_two_groups_async": two,
            "gpu_launches": main_leg["launches"],
            "clocks": main_leg["clocks"],
            "episode_stats": stats_all,
            "closed_loop": closed,
            "multi_agent": multi,
            "configs": configs,
        }
        if not args.no_cpu_baseline:   # rank 0, at every N (the other ranks wait at the barrier below)
            line["cpu_baseline"] = cpu_baseline_of(wl)
            line["cpu_baseline"]["reference_stack"] = reference_stack_baseline(300)
            if configs and "config3" in configs:   # the occupancy config's CPU cost is of a different order
                configs["config3"]["cpu_baseline"] = cpu_baseline_of(workload_of(3), budget_s=1.0)
        else:
            line["cpu_baseline"] = None
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    cx.barrier()
    if cx.world > 1:
        cx.dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
