"""The 'lidar_occupancy' Dreamer agent on one GPU: what the ConvEncoder costs and what collection runs at.  Prints (and
with --out writes) one JSON object.  Config 3: columbia, lidar_occupancy, action repeat 8, random weights of the
shipped RSSM / actor sizes with a depth-32 ConvEncoder (no trained encoder checkpoint ships with the project).

* the encode stage (rd_dreamer_encode_occupancy: k_conv1 + three k_dense implicit GEMMs, plus the hi + lo sum into the
  caller's embed buffer) and the full evaluation-mode agent step, in ms: CUDA events around `steps` calls on a fixed
  batch of images, warmed up, both precisions alternated, `reps` repetitions each
* closed-loop evaluation rollouts and recorded training rollouts (DeviceEpisodeStore), in env-steps/s
* the encoder's MACs and HBM bytes per env from its shapes, and the two lower bounds they give at the data-sheet rates
* the card's name, power limit and max SM clock, read in the same run
* --profile: the per-kernel split of the tf32x3 encode (torch.profiler, a pass of its own after the timed ones)

    python tools/dreamer_occupancy_bench.py [--envs 4096 16384] [--steps 50] [--reps 3] [--profile] [--out r13.json]
"""
import argparse
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(ROOT / "tests"))   # occupancy_reference: random weights with an encoder

from store_bench import card, config, timed  # noqa: E402

TF32_MAC_PER_S = 1125e12 / 2     # B200 data sheet, dense TF32, one GPU (FLOP = 2 MAC)
HBM_BYTES_PER_S = 7.7e12


def encoder_shapes(depth=32):
    """per env: valid and computed (padded-grid) tensor-core MACs of conv2..conv4, conv1's CUDA-core MACs, and the HBM
    bytes of one tf32x3 encode (u8 image in; every layer's hi + lo output written once and read once)"""
    layers, cin, size = [], 1, 64
    grids = (32, 16, 8, 2)   # the output grids the kernels compute on (conv1's includes its zeroed border)
    for l in range(4):
        cout, out = depth << l, (size - 4) // 2 + 1
        layers.append(dict(cin=cin, cout=cout, out=out, grid=grids[l], k=16 * cin))
        cin, size = cout, out
    valid = sum(L["out"] ** 2 * L["k"] * L["cout"] for L in layers[1:])
    padded = sum(L["grid"] ** 2 * L["k"] * L["cout"] for L in layers[1:])
    conv1 = layers[0]["out"] ** 2 * 16 * layers[0]["cout"]
    act = [L["grid"] ** 2 * L["cout"] * 4 * 2 for L in layers]    # hi + lo float32 on the stored grids
    act[-1] = 32 * depth * 4 * 2                                    # conv4 writes the compact embed
    hbm = 64 * 64 + 2 * sum(act[:-1]) + act[-1]
    return dict(layers=layers, tensor_macs_valid=valid, tensor_macs_computed=padded, conv1_macs=conv1,
                overcompute=padded / valid, hbm_bytes=hbm)


def bounds(shapes, n):
    return {"tf32x3_valid_ms": 3 * shapes["tensor_macs_valid"] * n / TF32_MAC_PER_S * 1e3,
            "tf32_valid_ms": shapes["tensor_macs_valid"] * n / TF32_MAC_PER_S * 1e3,
            "tf32x3_computed_ms": 3 * shapes["tensor_macs_computed"] * n / TF32_MAC_PER_S * 1e3,
            "hbm_ms": shapes["hbm_bytes"] * n / HBM_BYTES_PER_S * 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--capacity", type=int, default=260)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", action="store_true", help="add the per-kernel split of the tf32x3 encode (torch.profiler)")
    a = ap.parse_args()
    shapes = encoder_shapes()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("dreamer_occupancy_bench needs a CUDA device")
    torch.cuda.set_device(0)
    import occupancy_reference as occref
    from racing_dreamer_b200 import BatchedRaceEnv, DreamerPolicy
    from racing_dreamer_b200.episodes import DeviceEpisodeStore
    w = occref.random_weights(13)
    res = {"card": card(), "config": {"track": "columbia", "obs_type": "lidar_occupancy", "action_repeat": 8,
                                      "agent": "random weights, shipped RSSM / actor sizes, ConvEncoder depth 32",
                                      "noise": "philox"},
           "encoder_per_env": shapes, "runs": {}}
    tracks = ("columbia",)
    for n in a.envs:
        r = res["runs"][str(n)] = {"lower_bounds_ms": bounds(shapes, n)}
        # 1. encode stage and agent step, precisions alternated
        env = BatchedRaceEnv(config(tracks, n, "lidar_occupancy"), device="cuda:0")
        env.reset()
        occ = env.buf["occupancy"].clone()
        pols = {}
        for prec in ("tf32x3", "tf32"):
            pols[prec] = DreamerPolicy(BatchedRaceEnv(config(tracks, n, "lidar_occupancy"), device="cuda:0"), w,
                                       noise="philox", precision=prec)
            pols[prec].env.reset()
        emb = torch.empty((n, 1024), dtype=torch.float32, device="cuda:0")

        def encode(p):
            for _ in range(a.steps):
                p.env._check(p.env.lib.rd_dreamer_encode_occupancy(p.env._handle, occ.data_ptr(), emb.data_ptr(),
                                                                   p.env._stream()))

        def step(p):
            for _ in range(a.steps):
                p.act(occupancy=occ)

        for p in pols.values():
            encode(p)
            step(p)
        times = {f"{what}_{prec}": [] for what in ("encode", "agent_step") for prec in pols}
        for _ in range(a.reps):
            for prec, p in pols.items():
                times[f"encode_{prec}"].append(timed(torch, lambda: encode(p)) / a.steps)
                times[f"agent_step_{prec}"].append(timed(torch, lambda: step(p)) / a.steps)
        r["ms"] = {k: {"runs": v, "min": min(v)} for k, v in times.items()}
        if a.profile:   # per-kernel split of the tf32x3 encode, in a pass of its own (after the timed ones)
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                encode(pols["tf32x3"])
                torch.cuda.synchronize()
            split = {}
            for ev in prof.key_averages():
                t = getattr(ev, "device_time_total", 0.0)
                if t > 0:
                    split[ev.key[:90]] = {"calls": ev.count, "ms_per_encode": t / 1e3 / a.steps}
            r["encode_tf32x3_kernels"] = split
        for p in pols.values():
            p.env.close()
        env.close()
        # 2. closed-loop evaluation rollouts and recorded training rollouts (tf32x3)
        rates = {"eval_rollout": [], "recorded_train_rollout": []}
        e1 = BatchedRaceEnv(config(tracks, n, "lidar_occupancy"), device="cuda:0")
        e1.reset()
        p1 = DreamerPolicy(e1, w, noise="philox")
        e2 = BatchedRaceEnv(config(tracks, n, "lidar_occupancy", auto_reset=False), device="cuda:0")
        s2 = DeviceEpisodeStore(e2, capacity_rows=a.capacity)
        p2 = DreamerPolicy(e2, w, noise="philox")
        s2.reset()
        p1.rollout(10)
        p2.rollout(10, training=True, store=s2)
        torch.cuda.synchronize()
        for _ in range(a.reps):
            rates["eval_rollout"].append(n * a.steps / (timed(torch, lambda: p1.rollout(a.steps)) / 1e3))
            rates["recorded_train_rollout"].append(
                n * a.steps / (timed(torch, lambda: p2.rollout(a.steps, training=True, store=s2)) / 1e3))
        r["env_steps_per_s"] = {k: {"runs": v, "max": max(v)} for k, v in rates.items()}
        r["env_steps_per_s"]["train_episodes_held"] = s2.info()["held"]
        e1.close()
        e2.close()
        enc = r["ms"]["encode_tf32x3"]["min"]
        lb = r["lower_bounds_ms"]
        r["encode_tf32x3_over_bounds"] = {"hbm": lb["hbm_ms"] / enc, "tensor_valid": lb["tf32x3_valid_ms"] / enc,
                                          "tensor_computed": lb["tf32x3_computed_ms"] / enc}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
