"""CPU restatement (NumPy) of the reference's Dreamer agent inference step -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this module; nothing under
racing_dreamer_b200/ does.

What it restates (SURVEY.md §8-f2), line by line:
  * RacingDreamer.action / _preprocess_lidar / postprocess_action  [REF ros_agent/models/dreamer/racing_dreamer.py:45-82]
  * RSSM.obs_step / img_step / get_feat                            [REF ros_agent/models/dreamer/models.py:57-90]
  * ActionDecoder.__call__ ('tanh_normal' and 'normalized_tanhtransformed_normal')  [REF models.py:307-346]
  * SampleDist.mode, TanhBijector._forward_log_det_jacobian       [REF ros_agent/helpers/tools.py:70-73, 142-144]
  * Module.load: a checkpoint is the pickled tuple of `self.variables` [REF ros_agent/helpers/tools.py:25-33]; the
    order below is the one found in the shipped files (ros_agent/checkpoints/*/{rssm,actor}.pkl), identified by shape.

Third-party pieces the reference calls and that are NOT in /root/reference (TensorFlow 2.x / Keras / TFP, versions
unpinned in ros_agent; dreamer/requirements.txt pins tensorflow 2.3.1 / tfp 0.11.1), restated from their published
definitions:
  * tf.keras.layers.Dense: act(x @ kernel + bias); tf.nn.elu: x if x > 0 else expm1(x); tf.nn.softplus: log1p(exp(x))
  * tf.keras.layers.GRUCell (TF2 default reset_after=True, bias shape (2, 3*units), gate order z | r | h):
        mx = x @ kernel + bias[0];  mh = h @ recurrent_kernel + bias[1]
        z = sigmoid(mx_z + mh_z);  r = sigmoid(mx_r + mh_r);  hh = tanh(mx_h + r * mh_h);  h' = z * h + (1 - z) * hh
  * tf.keras.layers.BatchNormalization (inference): (x - moving_mean) / sqrt(moving_var + 1e-3) * gamma + beta;
    (pickled order: moving_mean, moving_variance, gamma, beta -- see load_checkpoint)
  * tfd.Normal.log_prob; TransformedDistribution.log_prob(y) = base.log_prob(x) - fldj(x) with the cached pre-image x;
    tfd.Independent(., 1) sums over the action dimension; tf.argmax returns the first maximum.

PARITY UNPINNED against TensorFlow itself: TensorFlow is not installable here, the reference ships no golden vectors
for its agents, and both random draws (posterior sample, the 100 actor samples) come from TF's RNG.  The restatement
therefore takes the standard-normal draws as inputs.  tests/test_cpu_dreamer_policy.py cross-checks the GRU cell
against torch.nn.GRUCell (same published equations, different gate order) and the checkpoint layout by shape.
"""
from __future__ import annotations

import pathlib
import pickle
from typing import Dict, Optional, Tuple

import numpy as np

STOCH, DETER, HIDDEN = 30, 200, 200          # [REF racing_dreamer.py:20]
ACTOR_LAYERS, ACTOR_UNITS = 4, 400           # [REF racing_dreamer.py:22-26]
INIT_STD, MIN_STD, MEAN_SCALE = 5.0, 1e-4, 5.0   # [REF racing_dreamer.py:23; models.py:311]
N_SAMPLES = 100                              # [REF ros_agent/helpers/tools.py:55]
BN_EPS = 1e-3                                # tf.keras BatchNormalization default epsilon


def load_checkpoint(checkpoint_dir) -> Dict[str, np.ndarray]:
    """rssm.pkl + actor.pkl -> named float32 arrays [REF racing_dreamer.py:30-32; tools.py:30-33]."""
    d = pathlib.Path(checkpoint_dir)
    with open(d / "rssm.pkl", "rb") as f:
        r = pickle.load(f)
    with open(d / "actor.pkl", "rb") as f:
        a = pickle.load(f)
    if len(r) != 13 or len(a) not in (10, 14):
        raise ValueError(f"unexpected checkpoint layout: {len(r)} rssm / {len(a)} actor variables")
    w = dict(gru_kernel=r[0], gru_recurrent=r[1], gru_bias=r[2], img1_w=r[3], img1_b=r[4], img2_w=r[5], img2_b=r[6],
             img3_w=r[7], img3_b=r[8], obs1_w=r[9], obs1_b=r[10], obs2_w=r[11], obs2_b=r[12])
    for i in range(ACTOR_LAYERS):
        w[f"h{i}_w"], w[f"h{i}_b"] = a[2 * i], a[2 * i + 1]
    if len(a) == 14:   # 'normalized' head: hnorm's four variables sit before hout's (tf.Module orders by name); inside a
        # Keras layer the sorted attribute walk meets _non_trainable_weights (moving mean, moving variance) before
        # _trainable_weights (gamma, beta) -- and a[9] is the all-positive one of the first two, as a variance must be
        w["bn_mean"], w["bn_var"], w["bn_gamma"], w["bn_beta"] = a[8], a[9], a[10], a[11]
        w["hout_w"], w["hout_b"] = a[12], a[13]
    else:
        w["hout_w"], w["hout_b"] = a[8], a[9]
    return {k: np.asarray(v, np.float32) for k, v in w.items()}


def n_actor_layers(w) -> int:
    """Trunk layers of a weight dict: h0_w, h1_w, ... (the shipped agents have ACTOR_LAYERS)."""
    return sum(1 for k in w if k.startswith("h") and k.endswith("_w") and k[1:-2].isdigit())


def random_weights(seed: int, n_beams: int = 1080, normalized: bool = False, actor_layers: int = ACTOR_LAYERS,
                   deter: int = DETER, hidden: int = HIDDEN, units: int = ACTOR_UNITS) -> Dict[str, np.ndarray]:
    """Glorot-ish random weights (for tests on machines without the checkpoints), by default of the shipped
    architecture; other trunk depths and widths (deter, hidden, units, n_beams = embed) exercise the product's general
    paths.  The draws are made in one fixed order, so the default arguments give the same arrays whatever the others."""
    rng = np.random.RandomState(seed)

    def dense(i, o):
        return (rng.uniform(-1, 1, (i, o)) * np.sqrt(3.0 / i)).astype(np.float32), (rng.uniform(-0.1, 0.1, o)).astype(np.float32)

    w = {}
    w["gru_kernel"], _ = dense(hidden, 3 * deter)
    w["gru_recurrent"], _ = dense(deter, 3 * deter)
    w["gru_bias"] = rng.uniform(-0.1, 0.1, (2, 3 * deter)).astype(np.float32)
    w["img1_w"], w["img1_b"] = dense(STOCH + 2, hidden)
    w["img2_w"], w["img2_b"] = dense(deter, hidden)
    w["img3_w"], w["img3_b"] = dense(hidden, 2 * STOCH)
    w["obs1_w"], w["obs1_b"] = dense(deter + n_beams, hidden)
    w["obs2_w"], w["obs2_b"] = dense(hidden, 2 * STOCH)
    i = STOCH + deter
    for k in range(actor_layers):
        w[f"h{k}_w"], w[f"h{k}_b"] = dense(i, units)
        i = units
    w["hout_w"], w["hout_b"] = dense(units, 4)
    if normalized:
        w["bn_gamma"] = rng.uniform(0.5, 2.0, 4).astype(np.float32)
        w["bn_beta"] = rng.uniform(-0.5, 0.5, 4).astype(np.float32)
        w["bn_mean"] = rng.uniform(-0.5, 0.5, 4).astype(np.float32)
        w["bn_var"] = rng.uniform(0.5, 2.0, 4).astype(np.float32)
    return w


def _elu(x):
    return np.where(x > 0, x, np.expm1(np.minimum(x, 0)))


def _softplus(x):
    return np.logaddexp(0, x)


def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def preprocess_lidar(scan: np.ndarray) -> np.ndarray:
    """[REF racing_dreamer.py:45-52]"""
    lidar = np.clip(scan, 0.0, 15.0)
    lidar = (lidar - 0.0) / (15.0 - 0.0) - 0.5
    return lidar.astype("float32")


def gru_cell(w, x, h, dt):
    mx = x @ w["gru_kernel"].astype(dt) + w["gru_bias"][0].astype(dt)
    mh = h @ w["gru_recurrent"].astype(dt) + w["gru_bias"][1].astype(dt)
    n = h.shape[-1]
    z = _sigmoid(mx[..., :n] + mh[..., :n])
    r = _sigmoid(mx[..., n:2 * n] + mh[..., n:2 * n])
    hh = np.tanh(mx[..., 2 * n:] + r * mh[..., 2 * n:])
    return z * h + (1 - z) * hh


def obs_step(w, stoch, deter, prev_action, embed, eps_stoch, dtype=np.float64):
    """RSSM.obs_step [REF models.py:63-74]: (posterior mean, std, stoch, deter).  The prior's own sample (img2/img3)
    is discarded by obs_step's caller [REF racing_dreamer.py:76-78] and is not computed."""
    dt = dtype
    x = np.concatenate([stoch, prev_action], -1).astype(dt)
    x = _elu(x @ w["img1_w"].astype(dt) + w["img1_b"].astype(dt))            # img1 [REF models.py:79-80]
    deter = gru_cell(w, x, deter.astype(dt), dt)                             # self._cell [REF models.py:81-82]
    x = np.concatenate([deter, embed.astype(dt)], -1)                        # [REF models.py:66]
    x = _elu(x @ w["obs1_w"].astype(dt) + w["obs1_b"].astype(dt))
    x = x @ w["obs2_w"].astype(dt) + w["obs2_b"].astype(dt)
    mean, std = x[..., :STOCH], x[..., STOCH:]
    std = _softplus(std) + 0.1
    stoch = mean + std * eps_stoch.astype(dt)                                # MultivariateNormalDiag.sample
    return mean, std, stoch, deter


def actor_dist(w, feat, dtype=np.float64):
    """ActionDecoder.__call__ -> (mean, std) of the pre-tanh Normal [REF models.py:320-346]."""
    dt = dtype
    x = feat.astype(dt)
    for i in range(n_actor_layers(w)):
        x = _elu(x @ w[f"h{i}_w"].astype(dt) + w[f"h{i}_b"].astype(dt))
    x = x @ w["hout_w"].astype(dt) + w["hout_b"].astype(dt)
    if "bn_gamma" in w:   # 'normalized_tanhtransformed_normal' [REF models.py:335-346], training=False
        x = (x - w["bn_mean"].astype(dt)) / np.sqrt(w["bn_var"].astype(dt) + BN_EPS) * w["bn_gamma"].astype(dt) + w["bn_beta"].astype(dt)
        mean, std = x[..., :2], x[..., 2:]
        std = _softplus(std) + MIN_STD
    else:                 # 'tanh_normal' [REF models.py:323-333]
        raw_init_std = np.log(np.exp(INIT_STD) - 1)
        mean, std = x[..., :2], x[..., 2:]
        mean = MEAN_SCALE * np.tanh(mean / MEAN_SCALE)
        std = _softplus(std + raw_init_std) + MIN_STD
    return mean, std


def sample_log_prob(mean, std, eps):
    """log_prob of tanh(mean + std * eps) under Independent(Transformed(Normal(mean, std), Tanh), 1); eps [..., S, 2]."""
    u = mean[..., None, :] + std[..., None, :] * eps
    base = -0.5 * eps ** 2 - np.log(std[..., None, :]) - 0.5 * np.log(2 * np.pi)
    fldj = 2.0 * (np.log(2.0) - u - _softplus(-2.0 * u))                     # [REF tools.py:142-144]
    return u, (base - fldj).sum(-1)


def mode(mean, std, eps_actor):
    """SampleDist.mode [REF tools.py:70-73]: the sample with the largest log_prob.  eps_actor: [N, S, 2] draws, or None
    for the zero-noise variant (the single 'sample' u = mean)."""
    if eps_actor is None:
        eps_actor = np.zeros(mean.shape[:-1] + (1, 2), mean.dtype)
    u, lp = sample_log_prob(mean, std, eps_actor.astype(mean.dtype))
    idx = np.argmax(lp, -1)
    best_u = np.take_along_axis(u, idx[..., None, None], -2)[..., 0, :]
    return np.tanh(best_u), np.take_along_axis(lp, idx[..., None], -1)[..., 0], idx, lp


def policy_step(w, scan, state: Optional[Tuple[np.ndarray, np.ndarray, np.ndarray]], eps_stoch, eps_actor, dtype=np.float64):
    """RacingDreamer.action for a batch [REF racing_dreamer.py:62-82].  state = (stoch, deter, action) or None (zeros,
    deter as wide as the weights' GRU).  Returns (agent-facing action in [-1, 1], new state, diagnostics)."""
    n = scan.shape[0]
    embed = preprocess_lidar(scan)
    if state is None:
        d = w["gru_recurrent"].shape[0]
        stoch, deter, action = np.zeros((n, STOCH), dtype), np.zeros((n, d), dtype), np.zeros((n, 2), dtype)
    else:
        stoch, deter, action = state
    mean, std, stoch, deter = obs_step(w, stoch, deter, action, embed, eps_stoch, dtype)
    feat = np.concatenate([stoch, deter], -1)                                # get_feat [REF models.py:57-58]
    amean, astd = actor_dist(w, feat, dtype)
    act, logp, idx, lp_all = mode(amean, astd, eps_actor)
    return act, (stoch, deter, act), dict(mean=mean, std=std, actor_mean=amean, actor_std=astd, logp=logp, index=idx, logp_all=lp_all)


def postprocess_action(action):
    """[REF racing_dreamer.py:54-60]: what the env's own action rescale (k_step prologue) computes."""
    action = np.clip(action, -1, +1)
    low, high = np.array([0.005, -1.0]), np.array([1.0, 1.0])
    return (action + 1) / 2 * (high - low) + low
