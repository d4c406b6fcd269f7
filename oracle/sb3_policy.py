"""Float64 restatement of the model-free baselines' actors: Stable-Baselines3's SAC actor and the actor half of its
ActorCriticPolicy (PPO / A2C), what ``Sb3Policy`` / ``rd_policy_mlp`` compute on the device.

The arithmetic is plain Linear + activation layers (checked in the CPU tests against ``torch.nn`` modules built from the
same state dict, in float64).  The SB3-specific composition is [UPSTREAM-RECALL: stable_baselines3 sac/policies.py
Actor, common/distributions.py SquashedDiagGaussianDistribution / DiagGaussianDistribution, common/policies.py
ActorCriticPolicy, common/torch_layers.py MlpExtractor -- SB3 1.x / 2.x]:

* SAC: latent = latent_pi(obs) (Linear + ReLU by default); mean = mu(latent); log_std = clamp(log_std(latent), -20, 2);
  action = tanh(mean + exp(log_std) e), e = 0 for the deterministic action.
* PPO / A2C: latent = policy_net(shared_net(obs)) (Linear + Tanh by default); mean = action_net(latent); log_std is a
  state-independent parameter; action = mean + exp(log_std) e, unclipped (the rollout buffer keeps it unclipped).

Weights use the canonical names of ``racing_dreamer_b200.policy.load_sb3_checkpoint``: w0, b0, ... (PyTorch layout
[out][in]), mean_w, mean_b, and log_std_w, log_std_b (SAC) or log_std (PPO).
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import numpy as np

LOG_STD_MIN, LOG_STD_MAX = -20.0, 2.0


def _linear(rng, out: int, inp: int, scale: float = 1.0):
    """nn.Linear's default initialisation: uniform(-1/sqrt(in), 1/sqrt(in)) for weight and bias, float32"""
    b = scale / np.sqrt(inp)
    return (rng.uniform(-b, b, (out, inp)).astype(np.float32), rng.uniform(-b, b, (out,)).astype(np.float32))


def sac_state_dict(seed: int, n_beams: int = 1080, widths: Sequence[int] = (256, 256), log_std_bias: float = -1.0,
                   critic: bool = True, scale: float = 1.0) -> Dict[str, np.ndarray]:
    """A SACPolicy state dict (key names and shapes of SB3's), with nn.Linear-style random weights and the critic's
    keys, which the actor ignores.  log_std_bias shifts the log_std head (SB3's initial std is ~1); scale multiplies
    the trunk's weights and biases (saturated tanh, dead relu units, activations beyond the init's range)."""
    rng = np.random.default_rng(seed)
    sd, prev = {}, n_beams
    for i, u in enumerate(widths):
        sd[f"actor.latent_pi.{2 * i}.weight"], sd[f"actor.latent_pi.{2 * i}.bias"] = _linear(rng, u, prev, scale)
        prev = u
    sd["actor.mu.weight"], sd["actor.mu.bias"] = _linear(rng, 2, prev)
    sd["actor.log_std.weight"], sd["actor.log_std.bias"] = _linear(rng, 2, prev)
    sd["actor.log_std.bias"] = (sd["actor.log_std.bias"] + np.float32(log_std_bias)).astype(np.float32)
    if critic:
        for q in range(2):
            for net in ("critic", "critic_target"):
                sd[f"{net}.qf{q}.0.weight"], sd[f"{net}.qf{q}.0.bias"] = _linear(rng, 8, n_beams + 2)
                sd[f"{net}.qf{q}.2.weight"], sd[f"{net}.qf{q}.2.bias"] = _linear(rng, 1, 8)
    return sd


def ppo_state_dict(seed: int, n_beams: int = 1080, widths: Sequence[int] = (64, 64), shared: Sequence[int] = (),
                   log_std: Sequence[float] = (-0.5, 0.25), critic: bool = True, scale: float = 1.0) -> Dict[str, np.ndarray]:
    """An ActorCriticPolicy state dict: ``shared`` widths under mlp_extractor.shared_net (older SB3), ``widths`` under
    mlp_extractor.policy_net, action_net, log_std, and the value side, which the actor ignores.  scale multiplies the
    actor trunk's weights and biases, as in sac_state_dict."""
    rng = np.random.default_rng(seed)
    sd, prev = {}, n_beams
    for i, u in enumerate(shared):
        sd[f"mlp_extractor.shared_net.{2 * i}.weight"], sd[f"mlp_extractor.shared_net.{2 * i}.bias"] = _linear(
            rng, u, prev, scale)
        prev = u
    trunk_in = prev
    for i, u in enumerate(widths):
        sd[f"mlp_extractor.policy_net.{2 * i}.weight"], sd[f"mlp_extractor.policy_net.{2 * i}.bias"] = _linear(
            rng, u, prev, scale)
        prev = u
    sd["action_net.weight"], sd["action_net.bias"] = _linear(rng, 2, prev)
    sd["log_std"] = np.asarray(log_std, np.float32)
    if critic:
        sd["mlp_extractor.value_net.0.weight"], sd["mlp_extractor.value_net.0.bias"] = _linear(rng, 16, trunk_in)
        sd["value_net.weight"], sd["value_net.bias"] = _linear(rng, 1, 16)
    return sd


def n_layers(w) -> int:
    return sum(1 for k in w if k[0] == "w" and k[1:].isdigit())


def actor(w, algo: str, activation: str, obs: np.ndarray, eps: Optional[np.ndarray] = None,
          deterministic: bool = True, dtype=np.float64, log_std_bounds=(LOG_STD_MIN, LOG_STD_MAX), matmul=None):
    """obs [N, n_beams] -> (mean [N, 2], std [N, 2], action [N, 2]) in `dtype`; eps [N, 2] standard normals
    (stochastic).  dtype=np.float32 is a float32 evaluation (float32 weights, products, sums and activations), the
    yardstick of a float32-grade kernel.  log_std_bounds: the SAC head's clamp.  matmul(x, w) -> x w^T, the products
    of every Linear layer (default: in `dtype`; the tests pass emulations of tensor-core arithmetic)."""
    act = {"relu": lambda x: np.maximum(x, dtype(0)), "tanh": np.tanh}[activation]
    f = lambda k: np.asarray(w[k], dtype)   # noqa: E731
    mm = matmul or (lambda a, b: a @ b.T)
    x = np.asarray(obs, dtype)
    for i in range(n_layers(w)):
        x = act(mm(x, f(f"w{i}")) + f(f"b{i}"))
    mean = mm(x, f("mean_w")) + f("mean_b")
    if algo == "sac":
        log_std = np.clip(mm(x, f("log_std_w")) + f("log_std_b"), dtype(log_std_bounds[0]), dtype(log_std_bounds[1]))
    else:
        log_std = np.broadcast_to(f("log_std"), mean.shape)
    std = np.exp(log_std)
    u = mean if deterministic or eps is None else mean + std * np.asarray(eps, dtype)
    return mean, std, (np.tanh(u) if algo == "sac" else u)


def random_actions(philox, seed: int, n: int, step: int, tag: int, gid0: int = 0) -> np.ndarray:
    """RandomPolicy's law: Philox4x32-10 block (gid0 + env, step, 0, tag) keyed (seed_lo, seed_hi ^ tag),
    a_k = 2 (x_k >> 8) 2^-24 - 1 (exact in float32).  philox: a vectorised Philox4x32-10 (counter arrays, key ints)."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    x = philox(np.arange(n) + gid0, step, 0, tag, seed & 0xFFFFFFFF, (seed >> 32) ^ tag)
    u = np.stack([(x[0] >> 8), (x[1] >> 8)], -1).astype(np.float64) / 16777216.0
    return (2.0 * u - 1.0).astype(np.float32)
