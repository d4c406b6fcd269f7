"""Float64 restatement of the 'lidar_occupancy' Dreamer agent -- TEST INFRASTRUCTURE ONLY (the tests and
tools/dreamer_occupancy_bench.py import it).  It extends oracle/dreamer_policy.py, whose RSSM and actor it reuses as
they are, with the image encoder:

  * ConvEncoder [UPSTREAM-RECALL: danijar Dreamer / racing_dreamer dreamer/models.py ConvEncoder; not in the reference
    tree]: the u8 image [N,64,64,1] cast to float (no scaling, SURVEY a11 [REF dreamer/tools.py:267-284]), four
    tf.keras Conv2D(depth * 2^l, kernel 4, stride 2, 'valid', relu) layers (kernels [kh][kw][Cin][Cout], biases
    [Cout]), the [N,2,2,8 depth] output flattened in (y, x, c) order to the embed (32 depth floats) obs1 reads.
"""
from typing import Dict, Optional, Tuple

import numpy as np

from oracle import dreamer_policy as dp

ENC_KEYS = tuple(f"enc{l}_{p}" for l in range(1, 5) for p in "wb")


def random_weights(seed: int, conv_depth: int = 32, normalized: bool = False, **kw) -> Dict[str, np.ndarray]:
    """dp.random_weights of an agent whose embed is 32 conv_depth (obs1_w [deter + 32 conv_depth][hidden]), plus the
    ConvEncoder's enc1_w, enc1_b .. enc4_w, enc4_b: He-uniform kernels (the ReLU stack keeps its scale), biases in
    [-0.1, 0.1], from a generator of their own so that the other arrays are dp.random_weights' draws."""
    w = dp.random_weights(seed, n_beams=32 * conv_depth, normalized=normalized, **kw)
    rng = np.random.RandomState([seed, 0x656E63])
    cin = 1
    for l in range(4):
        cout = conv_depth << l
        w[f"enc{l + 1}_w"] = (rng.uniform(-1, 1, (4, 4, cin, cout)) * np.sqrt(6.0 / (16 * cin))).astype(np.float32)
        w[f"enc{l + 1}_b"] = rng.uniform(-0.1, 0.1, cout).astype(np.float32)
        cin = cout
    return w


def conv_encoder(w, occ, dtype=np.float64):
    """ConvEncoder (module docstring) of u8 images [N,64,64] or [N,64,64,1] -> embed [N, 32 depth] in `dtype`."""
    dt = dtype
    x = np.asarray(occ).reshape(len(occ), 64, 64, 1).astype(dt)
    for l in range(4):
        k, b = w[f"enc{l + 1}_w"].astype(dt), w[f"enc{l + 1}_b"].astype(dt)
        ho, wo = (x.shape[1] - 4) // 2 + 1, (x.shape[2] - 4) // 2 + 1
        acc = np.zeros((x.shape[0], ho, wo, k.shape[3]), dt)
        for ky in range(4):
            for kx in range(4):
                acc += x[:, ky:ky + 2 * ho - 1:2, kx:kx + 2 * wo - 1:2, :] @ k[ky, kx]
        x = np.maximum(acc + b, 0)
    return x.reshape(x.shape[0], -1)


def policy_step(w, occ, state: Optional[Tuple[np.ndarray, np.ndarray, np.ndarray]], eps_stoch, eps_actor,
                dtype=np.float64, embed=None):
    """dp.policy_step with the ConvEncoder's embed of `occ` in place of _preprocess_lidar's (or `embed` as given)."""
    n = len(occ)
    if embed is None:
        embed = conv_encoder(w, occ, dtype)
    if state is None:
        d = w["gru_recurrent"].shape[0]
        stoch, deter, action = np.zeros((n, dp.STOCH), dtype), np.zeros((n, d), dtype), np.zeros((n, 2), dtype)
    else:
        stoch, deter, action = state
    mean, std, stoch, deter = dp.obs_step(w, stoch, deter, action, embed, eps_stoch, dtype)
    feat = np.concatenate([stoch, deter], -1)
    amean, astd = dp.actor_dist(w, feat, dtype)
    act, logp, idx, lp_all = dp.mode(amean, astd, eps_actor)
    return act, (stoch, deter, act), dict(mean=mean, std=std, actor_mean=amean, actor_std=astd, logp=logp, index=idx,
                                          logp_all=lp_all)
