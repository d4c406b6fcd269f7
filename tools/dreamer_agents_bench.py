"""Several Dreamer agents in one env batch on one GPU: what one batch of G agents costs against one agent, and against
today's alternative of G env handles with a policy each.  Prints (and with --out writes) one JSON object.  Config 2:
austria, 4096 envs, action repeat 8, tf32x3, Philox draws; agent 0 is the shipped austria_dreamer, the others random
weights of its architecture (the arithmetic per env is the same whatever the values).

* agent-step time in ms for the whole batch: CUDA events around `steps` agent steps on a fixed scan, warmed up, the arms
  alternated, `reps` repetitions each:
    one_agent                 DreamerPolicy on 4096 envs (today's policy)
    four_agents_contiguous    DreamerAgents, 4 agents on contiguous ranges of 1024 envs
    four_agents_by_slot       DreamerAgents, agent = car slot, agents_per_world = 4
    four_handles              4 env handles of 1024 envs, each with its own DreamerPolicy (the 4 steps back to back)
* closed-loop evaluation rollouts (agent step -> env step) of the slot-assigned DreamerAgents in 4-car worlds, and of one
  agent on the same env, in env-steps/s, alternated
* the card's name, power limit and max SM clock, read in the same run

    python tools/dreamer_agents_bench.py [--envs 4096] [--steps 100] [--reps 3] [--out r14_dreamer_agents_bench.json]
"""
import argparse
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from store_bench import card, config, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("dreamer_agents_bench needs a CUDA device")
    torch.cuda.set_device(0)
    from oracle import dreamer_policy as dp
    from racing_dreamer_b200 import BatchedRaceEnv, DreamerAgents, DreamerPolicy
    from racing_dreamer_b200.policy import load_dreamer_checkpoint
    n, steps, G = a.envs, a.steps, 4
    ws = [load_dreamer_checkpoint("austria_dreamer")] + [dp.random_weights(100 + g) for g in range(1, G)]
    res = {"card": card(), "config": {"track": "austria", "envs": n, "action_repeat": 8, "agents": G,
                                      "weights": "austria_dreamer + 3 random sets of its architecture",
                                      "precision": "tf32x3", "noise": "philox", "steps": steps, "reps": a.reps}}

    def cfg(envs, worlds=1):
        c = config(("austria",), envs)
        c.agents_per_world = worlds
        return c

    # arms: a list of (policy, scans) stepped back to back per timed agent step
    arms = {}
    env1 = BatchedRaceEnv(cfg(n), device="cuda:0")
    arms["one_agent"] = [(DreamerPolicy(env1, ws[0]), env1.reset()["lidar"].clone())]
    env2 = BatchedRaceEnv(cfg(n), device="cuda:0")
    contiguous = (np.arange(n) * G // n).astype(np.int32)
    arms["four_agents_contiguous"] = [(DreamerAgents(env2, ws, contiguous), env2.reset()["lidar"].clone())]
    env3 = BatchedRaceEnv(cfg(n, 4), device="cuda:0")
    by_slot = (np.arange(n) % 4).astype(np.int32)
    arms["four_agents_by_slot"] = [(DreamerAgents(env3, ws, by_slot), env3.reset()["lidar"].clone())]
    handles = [BatchedRaceEnv(cfg(n // G), device="cuda:0") for _ in range(G)]
    arms["four_handles"] = [(DreamerPolicy(e, ws[g]), e.reset()["lidar"].clone()) for g, e in enumerate(handles)]

    def step_ms(arm, k):
        return timed(torch, lambda: [pol.act(scans) for _ in range(k) for pol, scans in arm]) / k

    for arm in arms.values():
        step_ms(arm, 20)
    times = {k: [] for k in arms}
    for _ in range(a.reps):
        for k, arm in arms.items():
            times[k].append(step_ms(arm, steps))
    res["agent_step_ms"] = {k: {"runs": v, "min": min(v)} for k, v in times.items()}
    best = {k: min(v) for k, v in times.items()}
    res["agent_step_ratios"] = {k: best[k] / best["one_agent"] for k in best}
    res["one_batch_of_four_beats_four_handles"] = best["four_agents_by_slot"] < best["four_handles"] and \
        best["four_agents_contiguous"] < best["four_handles"]

    # closed loop: slot-assigned agents in 4-car worlds vs one agent on the same env config, alternated
    loops = {"four_agents_by_slot": env3, "one_agent_4car_worlds": BatchedRaceEnv(cfg(n, 4), device="cuda:0")}
    pols = {"four_agents_by_slot": arms["four_agents_by_slot"][0][0],
            "one_agent_4car_worlds": DreamerPolicy(loops["one_agent_4car_worlds"], ws[0])}
    for k, e in loops.items():
        e.reset()
        pols[k].rollout(20)
    rates = {k: [] for k in loops}
    for _ in range(a.reps):
        for k in loops:
            ms = timed(torch, lambda: pols[k].rollout(steps))
            rates[k].append(n * steps / (ms / 1e3))
    res["closed_loop_env_steps_per_s"] = {k: {"runs": v, "max": max(v)} for k, v in rates.items()}
    for e in [env1, env2, env3, loops["one_agent_4car_worlds"]] + handles:
        e.close()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
