"""Training-mode Dreamer collection on one GPU: what the training head and the in-place weight refresh cost.  Prints
(and with --out writes) one JSON object.  Config 2: austria, 4096 envs, action repeat 8, shipped austria_dreamer agent.

* agent-step time, evaluation (SampleDist.mode over 100 draws) vs training (one sample + exploration) head: CUDA
  events around `steps` agent steps on a fixed scan, the two modes alternated, `reps` repetitions each
* recorded Dreamer rollouts (DeviceEpisodeStore) in env-steps/s, training vs evaluation mode, alternated
* load_weights from CUDA tensors (packed on the device) vs building a fresh DreamerPolicy from host arrays
* the card's name, power limit and max SM clock, read in the same run

    python tools/dreamer_train_bench.py [--envs 4096] [--steps 100] [--reps 3] [--out dreamer_train_bench.json]
"""
import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from store_bench import card, config, timed  # noqa: E402


def agent_step_ms(torch, pol, scans, training, steps):
    return timed(torch, lambda: [pol.act(scans, training=training) for _ in range(steps)]) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--capacity", type=int, default=260)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("dreamer_train_bench needs a CUDA device")
    torch.cuda.set_device(0)
    from racing_dreamer_b200 import BatchedRaceEnv, DreamerPolicy
    from racing_dreamer_b200.episodes import DeviceEpisodeStore
    from racing_dreamer_b200.policy import load_dreamer_checkpoint
    w = load_dreamer_checkpoint("austria_dreamer")
    n, steps = a.envs, a.steps
    res = {"card": card(), "config": {"track": "austria", "envs": n, "action_repeat": 8, "agent": "austria_dreamer",
                                      "precision": "tf32x3", "noise": "philox"}}

    # 1. agent step, eval vs train, alternated
    env = BatchedRaceEnv(config(("austria",), n), device="cuda:0")
    scans = env.reset()["lidar"].clone()
    pol = DreamerPolicy(env, w, noise="philox")
    for training in (False, True):
        agent_step_ms(torch, pol, scans, training, 20)
    times = {"eval": [], "train": []}
    for _ in range(a.reps):
        for mode in ("eval", "train"):
            times[mode].append(agent_step_ms(torch, pol, scans, mode == "train", steps))
    res["agent_step_ms"] = {k: {"runs": v, "min": min(v)} for k, v in times.items()}
    env.close()

    # 2. recorded rollouts, train vs eval, alternated (one env + store per mode, same seed)
    arms = {}
    for mode in ("eval", "train"):
        e = BatchedRaceEnv(config(("austria",), n, auto_reset=False), device="cuda:0")
        s = DeviceEpisodeStore(e, capacity_rows=a.capacity)
        p = DreamerPolicy(e, w, noise="philox")
        s.reset()
        p.rollout(10, store=s, training=mode == "train")
        torch.cuda.synchronize()
        arms[mode] = (e, s, p)
    rates = {"eval": [], "train": []}
    for _ in range(a.reps):
        for mode, (e, s, p) in arms.items():
            ms = timed(torch, lambda: p.rollout(steps, store=s, training=mode == "train"))
            rates[mode].append(n * steps / (ms / 1e3))
    res["recorded_rollout_env_steps_per_s"] = {k: {"runs": v, "max": max(v)} for k, v in rates.items()}
    res["recorded_rollout_env_steps_per_s"]["train_episodes_held"] = arms["train"][1].info()["held"]
    for e, _, _ in arms.values():
        e.close()

    # 3. weight refresh: load_weights from CUDA tensors vs a fresh policy from host arrays (host clock, synchronised)
    env = BatchedRaceEnv(config(("austria",), n), device="cuda:0")
    env.reset()
    pol = DreamerPolicy(env, w, noise="philox")
    w_dev = {k: torch.from_numpy(v).cuda() for k, v in w.items()}
    torch.cuda.synchronize()
    refresh, fresh, refresh_dev = [], [], []
    for _ in range(a.reps + 1):
        t0 = time.perf_counter()
        pol.load_weights(w_dev)
        torch.cuda.synchronize()
        refresh.append((time.perf_counter() - t0) * 1e3)
        refresh_dev.append(timed(torch, lambda: pol.load_weights(w_dev)))
        t0 = time.perf_counter()
        DreamerPolicy(env, w, noise="philox")
        torch.cuda.synchronize()
        fresh.append((time.perf_counter() - t0) * 1e3)
    res["weights_ms"] = {"load_weights_cuda_tensors": {"runs": refresh[1:], "min": min(refresh[1:])},
                         "load_weights_cuda_tensors_device_events": {"runs": refresh_dev[1:], "min": min(refresh_dev[1:])},
                         "fresh_policy_from_host_arrays": {"runs": fresh[1:], "min": min(fresh[1:])}}
    env.close()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
