#!/usr/bin/env python
"""Per-launch times of k_lidar and k_step over tracks and batch sizes, timed with rd_enable_timing."""
import json
import os
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from racing_dreamer_b200 import BatchedRaceEnv, EnvConfig  # noqa: E402


def run(track, n, steps=200):
    env = BatchedRaceEnv(EnvConfig(tracks=(track,), n_envs=n, action_repeat=8, auto_reset=True, reset_mode="random", seed=1,
                                   time_limit_steps=250), device="cuda:0")
    rng = np.random.RandomState(0)
    a = torch.from_numpy(np.stack([np.full(n, 0.6), 0.8 * np.sin(rng.uniform(0, 6.28, n))], 1).astype(np.float32)).cuda()
    env.reset()
    for _ in range(50):
        env.step_raw(a.data_ptr())
    env.enable_timing(True)
    env.read_timing(reset=True)
    for _ in range(steps):
        env.step_raw(a.data_ptr())
    t = env.read_timing(reset=True)
    env.close()
    return t["lidar_ms"] / t["lidar_launches"], t["step_ms"] / t["step_launches"]


if __name__ == "__main__":
    out = []
    spec = os.environ.get("RD_SWEEP")   # e.g. "austria:4096" = one point
    if spec:
        tr, nn = spec.split(":")
        grid = [(tr, int(nn))]
    else:
        grid = [(t, n) for t in ("austria", "columbia", "barcelona") for n in (4096, 16384)]
    for track, n in grid:
        try:
            l, s = run(track, n)
            out.append(dict(track=track, n=n, lidar_ms=l, step_ms=s, rays_per_s=n * 1080 / l * 1e3))
        except Exception as e:  # e.g. map too large for shared memory
            out.append(dict(track=track, n=n, error=str(e)[:100]))
        print(json.dumps(out[-1]), flush=True)
