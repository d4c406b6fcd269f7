"""The model-free baselines' actors on one GPU (Sb3Policy, RandomPolicy): what an actor step costs and what closed-loop
collection reaches, against the host-stepped path with a torch actor.  Prints (and with --out writes) one JSON object.
Env: the baselines chain (baselines_config) on austria, action repeat 4.

* agent step: CUDA events around `steps` stochastic actor steps on a fixed scan, SAC [256, 256] and PPO [64, 64]
  alternated, `reps` repetitions each, at every --envs size; with the multiply-adds and the least bytes it moves
* closed loop in env-steps/s: Sb3Policy.rollout (SAC [256, 256], sampled actions) without and with a
  DeviceEpisodeStore, RandomPolicy.rollout, and HostSteppedEnv driven by a torch nn.Sequential actor of the same weights
  on the same GPU (observations to the device, actions back to the host every step)
* --profile: the per-kernel split of the agent step from torch.profiler (a separate pass, after the timed ones)
* the card's name, power limit and max SM clock, read in the same run

    python tools/mlp_agent_bench.py [--envs 4096 16384] [--steps 100] [--reps 3] [--profile] [--out mlp_agent_bench.json]
"""
import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from store_bench import card, timed  # noqa: E402

ARCHS = {"sac_256_256": ("sac", (256, 256)), "ppo_64_64": ("ppo", (64, 64))}
N_BEAMS = 1080


def state_dict(algo, widths):
    from oracle import sb3_policy as sp
    return sp.sac_state_dict(0, N_BEAMS, widths) if algo == "sac" else sp.ppo_state_dict(0, N_BEAMS, widths)


def cost(algo, widths, n):
    """multiply-adds per step and the least bytes the step moves: the scan read, its hi / lo split written and read
    back, each layer's activations written and read (hi + lo), the weights once, the actions written"""
    dims = (N_BEAMS,) + tuple(widths)
    macs = sum(a * b for a, b in zip(dims[:-1], dims[1:])) + dims[-1] * (4 if algo == "sac" else 2)
    act_bytes = 4 * (N_BEAMS + 4 * N_BEAMS + 4 * sum(widths) + 4 + 2)
    w_bytes = 2 * 4 * (macs + sum(widths) + 4)
    return {"macs_per_env": macs, "tf32_flop": 3 * 2 * macs * n, "bytes": act_bytes * n + w_bytes}


def torch_actor(torch, sd, algo, widths):
    """the SB3 actor as torch modules on the GPU: the path of a host-stepped SB3 model"""
    nn = torch.nn
    prefix = "actor.latent_pi" if algo == "sac" else "mlp_extractor.policy_net"
    act = nn.ReLU if algo == "sac" else nn.Tanh
    layers, prev = [], N_BEAMS
    for i, u in enumerate(widths):
        lin = nn.Linear(prev, u)
        lin.load_state_dict({"weight": torch.from_numpy(sd[f"{prefix}.{2 * i}.weight"]),
                             "bias": torch.from_numpy(sd[f"{prefix}.{2 * i}.bias"])})
        layers += [lin, act()]
        prev = u
    head = nn.Linear(prev, 2)
    hk = "actor.mu" if algo == "sac" else "action_net"
    head.load_state_dict({"weight": torch.from_numpy(sd[hk + ".weight"]), "bias": torch.from_numpy(sd[hk + ".bias"])})
    m = nn.Sequential(*layers, head).cuda().eval()
    return (lambda x: torch.tanh(m(x))) if algo == "sac" else m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--loop-envs", type=int, default=4096)
    ap.add_argument("--loop-steps", type=int, default=200)
    ap.add_argument("--host-steps", type=int, default=50)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mlp_agent_bench needs a CUDA device")
    torch.cuda.set_device(0)
    from racing_dreamer_b200 import BatchedRaceEnv
    from racing_dreamer_b200.compat import baselines_config
    from racing_dreamer_b200.episodes import DeviceEpisodeStore
    from racing_dreamer_b200.host import HostSteppedEnv
    from racing_dreamer_b200.policy import RandomPolicy, Sb3Policy
    sds = {k: state_dict(*v) for k, v in ARCHS.items()}
    res = {"card": card(), "config": {"track": "austria", "action_repeat": 4, "env": "baselines_config(mode='train')",
                                      "precision": "tf32x3", "noise": "philox", "agent_step": "stochastic"}}

    # 1. agent step, SAC and PPO alternated, per batch size
    res["agent_step_ms"] = {}
    for n in a.envs:
        env = BatchedRaceEnv(baselines_config("austria", n, seed=1), device="cuda:0")
        scans = env.reset()["lidar"].clone()
        times = {k: [] for k in ARCHS}
        for rep in range(a.reps + 1):
            for k in ARCHS:
                pol = Sb3Policy(env, sds[k])   # one actor per handle: each init replaces the other
                ms = timed(torch, lambda: [pol.act(scans, deterministic=False) for _ in range(a.steps)]) / a.steps
                if rep:   # rep 0 warms every shape
                    times[k].append(ms)
        out = {}
        for k, (algo, widths) in ARCHS.items():
            c = cost(algo, widths, n)
            t = min(times[k])
            out[k] = {"runs": times[k], "min": t, **c, "tflops_achieved": c["tf32_flop"] / (t * 1e-3) / 1e12,
                      "gbytes_per_s_least": c["bytes"] / (t * 1e-3) / 1e9, "launches": 2 + len(widths) + 1}
        res["agent_step_ms"][str(n)] = out
        env.close()

    # 2. closed loop: device rollouts (SAC, sampled actions) without / with the store, random prefill, host-stepped torch
    n, steps = a.loop_envs, a.loop_steps
    loop = {}
    for rec in (False, True):
        env = BatchedRaceEnv(baselines_config("austria", n, seed=2, auto_reset=not rec), device="cuda:0")
        store = DeviceEpisodeStore(env, capacity_rows=600) if rec else None
        pol, rnd = Sb3Policy(env, sds["sac_256_256"]), RandomPolicy(env)
        (store.reset() if rec else env.reset())
        for name, run in (("sac_256_256", lambda: pol.rollout(steps, deterministic=False, store=store)),
                          ("random", lambda: rnd.rollout(steps, store=store))):
            run()
            ms = min(timed(torch, run) for _ in range(a.reps))
            loop[f"{name}{'_store' if rec else ''}"] = {"env_steps_per_s": n * steps / (ms * 1e-3), "ms_per_step": ms / steps}
        env.close()
    henv = HostSteppedEnv(baselines_config("austria", n, seed=2))
    actor = torch_actor(torch, sds["sac_256_256"], "sac", (256, 256))
    obs = henv.reset()

    def host_loop(k):
        nonlocal obs
        with torch.no_grad():
            for _ in range(k):
                x = torch.from_numpy(np.ascontiguousarray(obs["lidar"])).cuda(non_blocking=False)
                obs = henv.step(actor(x).cpu().numpy())
    host_loop(5)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    host_loop(a.host_steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    loop["host_stepped_torch_sac_256_256"] = {"env_steps_per_s": n * a.host_steps / dt, "ms_per_step": 1e3 * dt / a.host_steps}
    henv.close()
    res["closed_loop"] = {"envs": n, "steps": steps, **loop}

    # 3. per-kernel split (separate pass: tracing slows the host)
    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        env = BatchedRaceEnv(baselines_config("austria", a.envs[0], seed=1), device="cuda:0")
        scans = env.reset()["lidar"].clone()
        split = {}
        for k in ARCHS:
            pol = Sb3Policy(env, sds[k])
            for _ in range(10):
                pol.act(scans, deterministic=False)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(a.steps):
                    pol.act(scans, deterministic=False)
                torch.cuda.synchronize()
            rows = {}
            for e in prof.key_averages():
                us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                if us and e.count:
                    rows[e.key[:120]] = {"us_per_step": us / a.steps, "calls": e.count}
            split[k] = rows
        res["kernel_split_envs"] = a.envs[0]
        res["kernel_split"] = split
        env.close()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
