"""On-device policies for closed-loop rollouts (SURVEY.md §8-f2).

``GapFollowerPolicy`` is the reference's follow-the-gap controller
[REF ros_agent/agents/follow_the_gap/src/agent.py:60-238] run for every env of a ``BatchedRaceEnv`` by the CUDA kernel
``k_gap_follower`` behind ``rd_policy_gap_follower`` (include/rd_env.h): scans are read where ``k_lidar`` wrote them and
the actions are written where ``k_step`` reads them, so ``rollout(n)`` advances the whole batch ``n`` steps without a
host round trip.  One controller per env; its state (PID memory, the node's two first-message gates) is cleared by the
env kernels whenever that env is reset.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch

from . import _abi
from .env import BatchedRaceEnv


def _check_store(env: BatchedRaceEnv, store) -> None:
    if getattr(store, "env", None) is not env:
        raise ValueError("store must be a DeviceEpisodeStore of this policy's env")


class GapFollowerPolicy:
    def __init__(self, env: BatchedRaceEnv, **overrides):
        """overrides: fields of ``rd_gap_follower`` (e.g. ``speed_scale=0.6``, ``kp=1.2``)."""
        self.env = env
        g = _abi.RdGapFollower()
        env.lib.rd_gap_follower_defaults(C.byref(env.cfg), C.byref(g))
        for k, v in overrides.items():
            if not hasattr(g, k):
                raise TypeError(f"unknown gap-follower parameter {k!r}")
            setattr(g, k, v)
        self.params = g
        with torch.cuda.device(env.device):
            env._check(env.lib.rd_policy_gap_follower_init(env._handle, C.byref(g)))
        self.actions = torch.zeros((env.n, 2), dtype=torch.float32, device=env.device)
        self.debug = torch.zeros((env.n, 4), dtype=torch.float64, device=env.device)

    def reset(self) -> None:
        """Clears every controller (env resets do this per env on the device already)."""
        with torch.cuda.device(self.env.device):
            self.env._check(self.env.lib.rd_policy_gap_follower_init(self.env._handle, C.byref(self.params)))

    def act(self, lidar: Optional[torch.Tensor] = None, speed: Optional[torch.Tensor] = None,
            debug: bool = False) -> torch.Tensor:
        """lidar f32 [N, n_beams] metres (default: the env's current observation), speed f32 [N] (default: the env's own
        longitudinal speed) -> agent-facing actions f32 [N, 2] (a persistent buffer)."""
        env = self.env
        li = env.buf["lidar"] if lidar is None else lidar
        if li.shape != (env.n, env.n_beams) or li.dtype != torch.float32 or li.device != env.device or not li.is_contiguous():
            raise ValueError(f"lidar must be a contiguous float32 CUDA tensor of shape ({env.n}, {env.n_beams})")
        sp = None
        if speed is not None:
            sp = speed.to(device=env.device, dtype=torch.float32).contiguous()
            if sp.shape != (env.n,):
                raise ValueError("speed must have shape (n_envs,)")
        with torch.cuda.device(env.device):
            env._check(env.lib.rd_policy_gap_follower(env._handle, li.data_ptr(), sp.data_ptr() if sp is not None else None,
                                                      self.actions.data_ptr(), self.debug.data_ptr() if debug else None,
                                                      env._stream()))
        return self.actions

    def rollout(self, n_steps: int, store=None):
        """n_steps x (controller -> env.step) enqueued on the current stream; returns the env's (obs, reward, done, info)
        views of the LAST step.  Episode statistics accumulate on the device (env.read_stats()).
        store: a ``DeviceEpisodeStore`` of this env -- every step is recorded and the finished envs are reset
        (``store.step``), still with no host synchronisation."""
        env = self.env
        with torch.cuda.device(env.device):
            if store is not None:
                _check_store(env, store)
                env._check(env.lib.rd_rollout_store(env._handle, _abi.STORE_POLICY_GAP_FOLLOWER, int(n_steps),
                                                    C.byref(env._out), self.actions.data_ptr(), 0, env._stream()))
            else:
                env._check(env.lib.rd_rollout_gap_follower(env._handle, int(n_steps), C.byref(env._out),
                                                           self.actions.data_ptr(), env._stream()))
        return env._obs(), env.buf["reward"], env.buf["done_bool"], env._info()

    def drive_command(self) -> Dict[str, torch.Tensor]:
        """The node's last published command per env (valid after ``act(debug=True)``)."""
        return {"steering_angle": self.debug[:, 0], "speed": self.debug[:, 1], "heading": self.debug[:, 2],
                "heading_distance": self.debug[:, 3]}


# ----------------------------------------------------------------------------------------------------------------------
# Dreamer agent (RSSM + actor) on the tensor cores
# ----------------------------------------------------------------------------------------------------------------------
import pathlib
import pickle

import numpy as np

CHECKPOINT_DIR = pathlib.Path(__file__).resolve().parent / "data" / "checkpoints"
_STOCH, _ACTOR_LAYERS = 30, 4   # [REF ros_agent/models/dreamer/racing_dreamer.py:20-26]


def load_dreamer_checkpoint(path) -> Dict[str, np.ndarray]:
    """A Dreamer agent's weights as named float32 arrays.

    ``path``: a directory holding the reference's ``rssm.pkl`` + ``actor.pkl`` (each the pickled tuple of the module's
    ``variables`` [REF ros_agent/helpers/tools.py:25-33; ros_agent/models/dreamer/racing_dreamer.py:30-32]), an ``.npz``
    written by ``save_dreamer_checkpoint``, or the name of a checkpoint packaged under ``data/checkpoints``.
    The variable order is the one of the shipped files (``ros_agent/checkpoints/*``): GRU kernel, recurrent kernel,
    bias; img1, img2, img3, obs1, obs2 (kernel, bias); actor h0..h3, [hnorm moving mean, moving variance, gamma, beta],
    hout.  img2/img3 (the prior head) are loaded but never evaluated by the agent step."""
    p = pathlib.Path(path)
    if not p.exists() and (CHECKPOINT_DIR / f"{path}.npz").exists():
        p = CHECKPOINT_DIR / f"{path}.npz"
    if p.is_file():
        with np.load(p) as z:
            return {k: np.ascontiguousarray(z[k], np.float32) for k in z.files}
    with open(p / "rssm.pkl", "rb") as f:
        r = pickle.load(f)
    with open(p / "actor.pkl", "rb") as f:
        a = pickle.load(f)
    if len(r) != 13 or len(a) not in (2 * _ACTOR_LAYERS + 2, 2 * _ACTOR_LAYERS + 6):
        raise ValueError(f"{p}: unexpected checkpoint layout ({len(r)} rssm / {len(a)} actor variables)")
    names = ["gru_kernel", "gru_recurrent", "gru_bias", "img1_w", "img1_b", "img2_w", "img2_b", "img3_w", "img3_b",
             "obs1_w", "obs1_b", "obs2_w", "obs2_b"]
    w = dict(zip(names, r))
    for i in range(_ACTOR_LAYERS):
        w[f"h{i}_w"], w[f"h{i}_b"] = a[2 * i], a[2 * i + 1]
    k = 2 * _ACTOR_LAYERS
    if len(a) == k + 6:   # actor_version 'normalized' [REF racing_dreamer.py:25-27]
        # tf.Module walks a Keras layer's attributes in sorted order and meets `_non_trainable_weights` (moving mean,
        # moving variance) before `_trainable_weights` (gamma, beta); in the shipped files the second array is the
        # only one of the first two that is all-positive, as a variance must be.
        w["bn_mean"], w["bn_var"], w["bn_gamma"], w["bn_beta"] = a[k:k + 4]
        k += 4
    w["hout_w"], w["hout_b"] = a[k], a[k + 1]
    return {n: np.ascontiguousarray(v, np.float32) for n, v in w.items()}


def save_dreamer_checkpoint(path, weights: Dict[str, np.ndarray]) -> None:
    np.savez_compressed(path, **{k: np.asarray(v, np.float32) for k, v in weights.items()})


def _dreamer_arch(w) -> tuple:
    """(deter, hidden, units, embed, layers, has_bn) of a weight dict (numpy arrays or tensors) whose names and shapes
    are the ones ``load_dreamer_checkpoint`` returns; ValueError otherwise."""
    for k in ("gru_kernel", "gru_recurrent", "gru_bias", "img1_w", "img1_b", "obs1_w", "obs1_b", "obs2_w", "obs2_b",
              "h0_w", "hout_w", "hout_b"):
        if k not in w:
            raise ValueError(f"checkpoint array {k} is missing")
    has_bn = "bn_gamma" in w
    if has_bn and any(k not in w for k in ("bn_beta", "bn_mean", "bn_var")):
        raise ValueError("checkpoint: bn_gamma without bn_beta / bn_mean / bn_var")
    deter = w["gru_recurrent"].shape[0]
    hidden = w["img1_w"].shape[1]
    units = w["h0_w"].shape[1]
    embed = w["obs1_w"].shape[0] - deter
    # the shipped agents have four trunk layers [REF racing_dreamer.py:22-26]; a weight dict may hold 1..7 (h0_w ...)
    layers = sum(1 for k in w if k.startswith("h") and k.endswith("_w") and k[1:-2].isdigit())
    if not 1 <= layers <= 7 or any(f"h{i}_w" not in w or f"h{i}_b" not in w for i in range(layers)):
        raise ValueError(f"actor trunk: expected h0_w/h0_b .. h{{k}}_w/h{{k}}_b for 1..7 layers, found {layers}")
    expect = {"gru_kernel": (hidden, 3 * deter), "gru_recurrent": (deter, 3 * deter), "gru_bias": (2, 3 * deter),
              "img1_w": (_STOCH + 2, hidden), "img1_b": (hidden,), "obs1_w": (deter + embed, hidden),
              "obs1_b": (hidden,), "obs2_w": (hidden, 2 * _STOCH), "obs2_b": (2 * _STOCH,),
              "h0_w": (_STOCH + deter, units), "hout_w": (units, 4), "hout_b": (4,)}
    expect.update({f"h{i}_w": (units, units) for i in range(1, layers)})
    expect.update({f"h{i}_b": (units,) for i in range(layers)})
    if has_bn:
        expect.update({k: (4,) for k in ("bn_gamma", "bn_beta", "bn_mean", "bn_var")})
    for k, shp in expect.items():
        if tuple(w[k].shape) != shp:
            raise ValueError(f"checkpoint array {k} has shape {tuple(w[k].shape)}, expected {shp}")
    return deter, hidden, units, embed, layers, has_bn


def exploration_amount(amount: float, decay: float, min_amount: float, env_steps: int) -> np.float32:
    """The exploration noise scale of a training step [REF dreamer/dreamer.py, Dreamer._exploration]: amount, times
    0.5 ** (env_steps / decay) if decay > 0, at least min_amount if min_amount > 0 -- in float64, rounded once to
    float32 (what rd_policy_dreamer_train applies)."""
    a = float(amount)
    if decay > 0:
        a *= 0.5 ** (float(env_steps) / float(decay))
    if min_amount > 0:
        a = max(float(min_amount), a)
    return np.float32(a)


def env_steps_per_training_step(cfg) -> int:
    """Dreamer's step counter advances by len(reset) * action_repeat per training call [REF dreamer/dreamer.py,
    Dreamer.__call__]: one row per car of the batch."""
    return int(cfg.n_envs) * int(cfg.action_repeat)


class DreamerPolicy:
    """The reference's ``RacingDreamer`` agent [REF ros_agent/models/dreamer/racing_dreamer.py:9-85] for every env of a
    ``BatchedRaceEnv``: ``_preprocess_lidar`` -> ``RSSM.obs_step`` -> ``ActionDecoder`` -> ``SampleDist.mode()``, nine
    launches of the tcgen05 kernel ``k_dense`` per agent step.  precision 'tf32x3' (default) evaluates every product as
    three TF32 tensor-core passes over hi/lo split float32 operands (float32-grade, like the reference's TensorFlow);
    'tf32' is a single pass (~1e-3 relative per layer).  The recurrent
    state lives on the device, one row per env, and is zeroed by the env kernels whenever that env is reset
    (``state=None`` in the reference).  ``act()`` returns agent-facing actions in [-1, 1]; the env's own action rescale
    is ``postprocess_action``.

    noise: 'philox' (default; the reference draws from TensorFlow's RNG), 'zero' (stoch = posterior mean,
    action = tanh(actor mean)) or 'explicit' (pass ``eps_stoch`` [N,30] and ``eps_actor`` [N,100,2] to ``act``).

    Training mode (``act(training=True)``, ``rollout(n, training=True)``) is ``Dreamer.policy(..., training=True)``
    [REF dreamer/dreamer.py]: one sample of the actor distribution instead of the mode, plus additive Gaussian
    exploration ``clip(a + amount * N(0, 1), -1, 1)``.  The amount is ``expl_amount``, halved every ``expl_decay`` env
    steps if ``expl_decay`` > 0 and floored at ``expl_min`` if ``expl_min`` > 0; ``env_steps`` counts
    ``n_envs * action_repeat`` per training step.  The defaults 0.3 / 0 / 0 are Dreamer's ``define_config`` values
    [UPSTREAM-RECALL].  ``load_weights`` hands the agent a learner's new weights without touching its state."""

    NOISE = {"zero": _abi.RD_NOISE_ZERO, "philox": _abi.RD_NOISE_PHILOX, "explicit": _abi.RD_NOISE_EXPLICIT}

    PRECISION = {"tf32x3": _abi.RD_PRECISION_TF32X3, "tf32": _abi.RD_PRECISION_TF32}

    def __init__(self, env: BatchedRaceEnv, checkpoint, actor_version: Optional[str] = None, noise: str = "philox",
                 n_samples: int = 100, precision: str = "tf32x3", expl_amount: float = 0.3, expl_decay: float = 0.0,
                 expl_min: float = 0.0):
        self.env = env
        w = checkpoint if isinstance(checkpoint, dict) else load_dreamer_checkpoint(checkpoint)
        w = {k: np.ascontiguousarray(v, np.float32) for k, v in w.items()}
        has_bn = "bn_gamma" in w
        if actor_version is None:
            actor_version = "normalized" if has_bn else "default"
        if actor_version not in ("default", "normalized"):
            raise NotImplementedError(f"actor version {actor_version} not implemented")   # [REF racing_dreamer.py:28-29]
        if (actor_version == "normalized") != has_bn:
            raise ValueError(f"actor_version {actor_version!r} does not match the checkpoint (hnorm variables "
                             f"{'present' if has_bn else 'absent'})")
        if noise not in self.NOISE:
            raise ValueError(f"noise {noise!r}: expected one of {sorted(self.NOISE)}")
        self.noise = noise
        self.weights = w
        self._arch = _dreamer_arch(w)
        deter, hidden, units, embed, layers, _ = self._arch
        if embed != env.n_beams:
            raise ValueError(f"the checkpoint embeds {embed} beams, the env casts {env.n_beams}")
        if precision not in self.PRECISION:
            raise ValueError(f"precision {precision!r}: expected one of {sorted(self.PRECISION)}")
        self.precision = precision
        self.n_samples, self.deter = int(n_samples), deter
        self._bn = None
        if has_bn:
            self._bn = np.ascontiguousarray(np.stack([w["bn_gamma"], w["bn_beta"], w["bn_mean"], w["bn_var"]]), np.float32)
        s = self._weights_struct(w, self._bn, lambda a: a.ctypes.data_as(C.c_void_p))
        with torch.cuda.device(env.device):
            env._check(env.lib.rd_policy_dreamer_init(env._handle, C.byref(s)))
        self.actions = torch.zeros((env.n, 2), dtype=torch.float32, device=env.device)
        self.debug = torch.zeros(env.n * _abi.RD_DREAMER_DEBUG_FLOATS, dtype=torch.float32, device=env.device)
        self.expl_amount, self.expl_decay, self.expl_min = float(expl_amount), float(expl_decay), float(expl_min)
        self._set_exploration(0)
        self._staged = None

    def _weights_struct(self, w, bn, ptr) -> "_abi.RdDreamerWeights":
        deter, hidden, units, embed, layers, _ = self._arch
        s = _abi.RdDreamerWeights()
        s.stoch, s.deter, s.hidden, s.embed, s.actor_units, s.actor_layers = _STOCH, deter, hidden, embed, units, layers
        for k in ("gru_kernel", "gru_recurrent", "gru_bias", "img1_w", "img1_b", "obs1_w", "obs1_b", "obs2_w", "obs2_b"):
            setattr(s, k, ptr(w[k]))
        for i in range(layers):
            s.actor_w[i], s.actor_b[i] = ptr(w[f"h{i}_w"]), ptr(w[f"h{i}_b"])
        s.actor_w[layers], s.actor_b[layers] = ptr(w["hout_w"]), ptr(w["hout_b"])
        if bn is not None:
            s.bn = ptr(bn)
        s.init_std, s.min_std, s.mean_scale, s.bn_eps = 5.0, 1e-4, 5.0, 1e-3   # [REF racing_dreamer.py:23; models.py:311]
        s.n_samples = self.n_samples                                            # [REF ros_agent/helpers/tools.py:55]
        s.precision = self.PRECISION[self.precision]
        return s

    def _set_exploration(self, env_steps: int) -> None:
        x = _abi.RdDreamerExploration(self.expl_amount, self.expl_decay, self.expl_min, int(env_steps))
        self.env._check(self.env.lib.rd_policy_dreamer_set_exploration(self.env._handle, C.byref(x)))

    @property
    def env_steps(self) -> int:
        """Dreamer's env-step counter of the exploration schedule (n_envs * action_repeat per training step)."""
        x = _abi.RdDreamerExploration()
        self.env._check(self.env.lib.rd_policy_dreamer_get_exploration(self.env._handle, C.byref(x)))
        return int(x.env_steps)

    @env_steps.setter
    def env_steps(self, value: int) -> None:
        if int(value) < 0:
            raise ValueError("env_steps must be >= 0")
        self._set_exploration(int(value))

    def exploration_amount(self) -> np.float32:
        """The exploration amount the next training step applies."""
        return exploration_amount(self.expl_amount, self.expl_decay, self.expl_min, self.env_steps)

    def load_weights(self, weights) -> None:
        """New weights for the agent, e.g. a learner's parameters after an update: a dict with the names and shapes
        ``load_dreamer_checkpoint`` returns, of numpy arrays or of tensors (CUDA tensors on the env's device are read
        there).  Everything is validated before any device work; the architecture and BN presence must be the ones
        the policy was built with.  The values are packed on the device on the current stream: steps enqueued before
        use the old weights, steps enqueued after the new ones, with no host synchronisation when the sources are
        CUDA tensors.  The recurrent state, the noise counter and ``env_steps`` are kept.  The sources stay referenced
        by the policy until the next call; writing to them afterwards on another stream needs the caller's ordering."""
        env = self.env
        if not isinstance(weights, dict):
            raise TypeError("weights must be a dict of arrays")
        arch = _dreamer_arch(weights)
        if arch != self._arch:
            names = ("deter", "hidden", "units", "embed", "actor layers", "BN head")
            diff = [f"{n} {a} != {b}" for n, a, b in zip(names, arch, self._arch) if a != b]
            raise ValueError("the weights do not match the policy's architecture: " + ", ".join(diff))
        layers = arch[4]
        keys = ["gru_kernel", "gru_recurrent", "gru_bias", "img1_w", "img1_b", "obs1_w", "obs1_b", "obs2_w", "obs2_b",
                "hout_w", "hout_b"] + [f"h{i}_{p}" for i in range(layers) for p in "wb"]
        if arch[5]:
            keys += ["bn_gamma", "bn_beta", "bn_mean", "bn_var"]
        on_device = False
        for k in keys:
            v = weights[k]
            if isinstance(v, torch.Tensor):
                if v.device.type != "cpu" and v.device != env.device:
                    raise ValueError(f"weight {k} is on {v.device}, the policy on {env.device}")
                on_device |= v.is_cuda
                if not v.dtype.is_floating_point:
                    raise ValueError(f"weight {k} has dtype {v.dtype}, expected a float dtype")
            elif not np.issubdtype(np.asarray(v).dtype, np.floating):
                raise ValueError(f"weight {k} has dtype {np.asarray(v).dtype}, expected a float dtype")
        if on_device:
            def dev(v):
                t = v.detach() if isinstance(v, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(v, np.float32))
                return t.to(device=env.device, dtype=torch.float32).contiguous()
            staged = {k: dev(weights[k]) for k in keys}
            bn = torch.stack([staged[k] for k in ("bn_gamma", "bn_beta", "bn_mean", "bn_var")]).contiguous() if arch[5] else None
            ptr = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731
        else:
            host = lambda v: v.detach().numpy() if isinstance(v, torch.Tensor) else v   # noqa: E731
            staged = {k: np.ascontiguousarray(host(weights[k]), np.float32) for k in keys}
            bn = np.ascontiguousarray(np.stack([staged[k] for k in ("bn_gamma", "bn_beta", "bn_mean", "bn_var")]),
                                      np.float32) if arch[5] else None
            ptr = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
        s = self._weights_struct(staged, bn, ptr)
        with torch.cuda.device(env.device):
            env._check(env.lib.rd_policy_dreamer_set_weights(env._handle, C.byref(s), int(on_device), env._stream()))
        self._staged = (staged, bn)

    def act(self, lidar: Optional[torch.Tensor] = None, eps_stoch: Optional[torch.Tensor] = None,
            eps_actor: Optional[torch.Tensor] = None, debug: bool = False, noise: Optional[str] = None,
            training: bool = False, eps_sample: Optional[torch.Tensor] = None,
            eps_expl: Optional[torch.Tensor] = None) -> torch.Tensor:
        """lidar f32 [N, n_beams] (default: the env's current observation) -> agent-facing actions f32 [N, 2].
        training=True: one actor sample plus exploration (the class docstring); noise='explicit' then takes
        ``eps_stoch`` [N,30], ``eps_sample`` [N,2] and ``eps_expl`` [N,2]."""
        env = self.env
        li = env.buf["lidar"] if lidar is None else lidar
        if li.shape != (env.n, env.n_beams) or li.dtype != torch.float32 or li.device != env.device or not li.is_contiguous():
            raise ValueError(f"lidar must be a contiguous float32 CUDA tensor of shape ({env.n}, {env.n_beams})")
        mode = self.NOISE[noise or self.noise]
        cast = lambda t: t.to(device=env.device, dtype=torch.float32).contiguous()   # noqa: E731
        es = ea = ex = None
        if mode == _abi.RD_NOISE_EXPLICIT and training:
            if eps_stoch is None or eps_sample is None or eps_expl is None:
                raise ValueError("training with noise='explicit' needs eps_stoch [N,30], eps_sample [N,2] and eps_expl [N,2]")
            es, ea, ex = cast(eps_stoch), cast(eps_sample), cast(eps_expl)
            if es.shape != (env.n, _STOCH) or ea.shape != (env.n, 2) or ex.shape != (env.n, 2):
                raise ValueError("eps_stoch must be [N,30], eps_sample and eps_expl [N,2]")
        elif mode == _abi.RD_NOISE_EXPLICIT:
            if eps_stoch is None or eps_actor is None:
                raise ValueError("noise='explicit' needs eps_stoch [N,30] and eps_actor [N,n_samples,2]")
            es, ea = cast(eps_stoch), cast(eps_actor)
            if es.shape != (env.n, _STOCH) or ea.shape != (env.n, self.n_samples, 2):
                raise ValueError("eps_stoch must be [N,30] and eps_actor [N,n_samples,2]")
        p = lambda t: t.data_ptr() if t is not None else None   # noqa: E731
        dbg = self.debug.data_ptr() if debug else None
        with torch.cuda.device(env.device):
            if training:
                env._check(env.lib.rd_policy_dreamer_train(env._handle, li.data_ptr(), self.actions.data_ptr(), mode,
                                                           p(es), p(ea), p(ex), dbg, env._stream()))
            else:
                env._check(env.lib.rd_policy_dreamer(env._handle, li.data_ptr(), self.actions.data_ptr(), mode,
                                                     p(es), p(ea), dbg, env._stream()))
        return self.actions

    def diagnostics(self) -> Dict[str, torch.Tensor]:
        """Valid after ``act(debug=True)``: posterior mean/std, actor mean/std, action, log-prob and index of the mode.
        After a training step: the sample before exploration, its log-prob and index 0."""
        n = self.env.n
        post = self.debug[: n * 2 * _STOCH].view(n, 2 * _STOCH)
        act = self.debug[n * 2 * _STOCH:].view(n, 8)
        return {"mean": post[:, :_STOCH], "std": post[:, _STOCH:], "actor_mean": act[:, 0:2], "actor_std": act[:, 2:4],
                "action": act[:, 4:6], "logp": act[:, 6], "index": act[:, 7]}

    def get_state(self):
        """(stoch [N,30], deter [N,deter], previous action [N,2]) -- the reference's ``state`` tuple."""
        env = self.env
        st = torch.empty((env.n, _STOCH), dtype=torch.float32, device=env.device)
        de = torch.empty((env.n, self.deter), dtype=torch.float32, device=env.device)
        ac = torch.empty((env.n, 2), dtype=torch.float32, device=env.device)
        with torch.cuda.device(env.device):
            env._check(env.lib.rd_policy_dreamer_get_state(env._handle, st.data_ptr(), de.data_ptr(), ac.data_ptr(), env._stream()))
        return st, de, ac

    def set_state(self, stoch=None, deter=None, action=None) -> None:
        env = self.env
        cast = lambda t, w: None if t is None else t.to(device=env.device, dtype=torch.float32).contiguous().view(env.n, w)  # noqa: E731
        st, de, ac = cast(stoch, _STOCH), cast(deter, self.deter), cast(action, 2)
        with torch.cuda.device(env.device):
            env._check(env.lib.rd_policy_dreamer_set_state(env._handle, st.data_ptr() if st is not None else None,
                                                           de.data_ptr() if de is not None else None,
                                                           ac.data_ptr() if ac is not None else None, env._stream()))

    def reset(self) -> None:
        """Zero every agent's recurrent state (env resets do this per env on the device already)."""
        z = lambda w: torch.zeros((self.env.n, w), dtype=torch.float32, device=self.env.device)   # noqa: E731
        self.set_state(z(_STOCH), z(self.deter), z(2))

    def rollout(self, n_steps: int, noise: Optional[str] = None, store=None, training: bool = False):
        """n_steps x (agent step -> env.step) enqueued on the current stream, no host round trip.  store: a
        ``DeviceEpisodeStore`` of this env that records every step and resets the finished envs (``store.step``).
        training=True: training-mode agent steps (sampled, explored actions; the recorded actions are the explored ones)."""
        env = self.env
        mode = self.NOISE[noise or self.noise]
        with torch.cuda.device(env.device):
            if store is not None:
                _check_store(env, store)
                policy = _abi.STORE_POLICY_DREAMER_TRAIN if training else _abi.STORE_POLICY_DREAMER
                env._check(env.lib.rd_rollout_store(env._handle, policy, int(n_steps), C.byref(env._out),
                                                    self.actions.data_ptr(), mode, env._stream()))
            else:
                run = env.lib.rd_rollout_dreamer_train if training else env.lib.rd_rollout_dreamer
                env._check(run(env._handle, int(n_steps), C.byref(env._out), self.actions.data_ptr(), mode, env._stream()))
        return env._obs(), env.buf["reward"], env.buf["done_bool"], env._info()
