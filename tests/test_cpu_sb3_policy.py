"""CPU: reading SB3 policies for the on-device model-free actors (load_sb3_checkpoint), the float64 restatement
oracle/sb3_policy.py against torch.nn itself, the random-action and MLP-noise Philox layouts, and the new ABI."""
import ctypes as C
import io
import json
import re
import zipfile
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import sb3_policy as sp
from racing_dreamer_b200 import _abi
from racing_dreamer_b200.policy import load_sb3_checkpoint
from test_cpu_dreamer_train import normal4
from test_cpu_episode_store import philox4x32_10

ROOT = Path(__file__).resolve().parents[1]
STREAM_MLP = 0x4D4C5041      # RD_STREAM_MLP
STREAM_RANDOM = 0x524E4441   # RD_STREAM_RANDOM


def mlp_normals(seed, n, step, gid0=0):
    """the Philox normals e [n, 2] of MLP actor step `step`: z0, z1 of block (gid, step, 0, RD_STREAM_MLP)"""
    return normal4(seed, np.arange(n) + gid0, step, 0, STREAM_MLP)[:, :2]


def random_actions(seed, n, step, gid0=0):
    return sp.random_actions(philox4x32_10, seed, n, step, STREAM_RANDOM, gid0)


def tensors(sd):
    return {k: torch.from_numpy(v) for k, v in sd.items()}


def write_zip(path, sd, policy_kwargs=None, data=True):
    """an SB3 model zip: policy.pth (torch.save of the state dict) and the `data` JSON"""
    buf = io.BytesIO()
    torch.save(tensors(sd), buf)
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
        if data:
            d = {"policy_class": {":type:": "<class 'abc.ABCMeta'>", ":serialized:": "gAWV"}}
            if policy_kwargs is not None:
                d["policy_kwargs"] = policy_kwargs
            z.writestr("data", json.dumps(d))
        z.writestr("_stable_baselines3_version", "2.3.0")
    return path


CASES = [("sac", dict(widths=(256, 256))), ("sac", dict(widths=(400, 300))), ("sac", dict(widths=(32,))),
         ("sac", dict(widths=(64, 48, 40, 36))), ("ppo", dict(widths=(64, 64))), ("ppo", dict(widths=(64, 64), shared=(64,))),
         ("ppo", dict(widths=(100,)))]


def make_sd(algo, seed=0, n_beams=1080, **kw):
    return sp.sac_state_dict(seed, n_beams, **kw) if algo == "sac" else sp.ppo_state_dict(seed, n_beams, **kw)


@pytest.mark.parametrize("algo,kw", CASES)
def test_parse_state_dicts(algo, kw):
    sd = make_sd(algo, 1, **kw)
    for src in (sd, tensors(sd)):
        a, w, meta = load_sb3_checkpoint(src, n_beams=1080)
        assert a == algo
        widths = tuple(kw.get("shared", ())) + tuple(kw["widths"])
        assert meta == {"activation": "relu" if algo == "sac" else "tanh", "widths": widths, "in_features": 1080}
        assert sp.n_layers(w) == len(widths)
        assert all(v.dtype == np.float32 and v.flags.c_contiguous for v in w.values())
        head = {"mean_w", "mean_b"} | ({"log_std_w", "log_std_b"} if algo == "sac" else {"log_std"})
        assert set(w) == {f"{p}{i}" for i in range(len(widths)) for p in "wb"} | head
        first = "actor.latent_pi.0.weight" if algo == "sac" else (
            "mlp_extractor.shared_net.0.weight" if "shared" in kw else "mlp_extractor.policy_net.0.weight")
        np.testing.assert_array_equal(w["w0"], sd[first])


@pytest.mark.parametrize("algo", ["sac", "ppo"])
def test_zip_round_trip(tmp_path, algo):
    sd = make_sd(algo, 2, widths=(64, 64))
    a, w, meta = load_sb3_checkpoint(write_zip(tmp_path / "m.zip", sd), n_beams=1080)
    assert a == algo and meta["activation"] == ("relu" if algo == "sac" else "tanh")
    _, w2, _ = load_sb3_checkpoint(sd)
    assert all(np.array_equal(w[k], w2[k]) for k in w)
    # activation_fn as SB3 writes a non-JSON policy_kwargs item: its str() next to the pickled dict
    pk = {":type:": "<class 'dict'>", ":serialized:": "gAWV", "net_arch": [64, 64],
          "activation_fn": "<class 'torch.nn.modules.activation.Tanh'>"}
    assert load_sb3_checkpoint(write_zip(tmp_path / "t.zip", sd, pk))[2]["activation"] == "tanh"
    pk["activation_fn"] = "<class 'torch.nn.modules.activation.ReLU'>"
    assert load_sb3_checkpoint(write_zip(tmp_path / "r.zip", sd, pk))[2]["activation"] == "relu"
    assert load_sb3_checkpoint(write_zip(tmp_path / "e.zip", sd, {}))[2]["activation"] == _default(algo)
    # activation= wins over what the zip says
    assert load_sb3_checkpoint(write_zip(tmp_path / "o.zip", sd, pk), activation="tanh")[2]["activation"] == "tanh"
    # a bare policy.pth
    torch.save(tensors(sd), tmp_path / "policy.pth")
    assert load_sb3_checkpoint(tmp_path / "policy.pth")[0] == algo


def _default(algo):
    return "relu" if algo == "sac" else "tanh"


def test_zip_activation_unreadable(tmp_path):
    sd = make_sd("sac", 3, widths=(32,))
    pk = {":type:": "<class 'dict'>", ":serialized:": "gAWV"}
    with pytest.raises(ValueError, match="activation="):
        load_sb3_checkpoint(write_zip(tmp_path / "u.zip", sd, pk))
    assert load_sb3_checkpoint(write_zip(tmp_path / "u2.zip", sd, pk), activation="relu")[2]["activation"] == "relu"
    pk = {":type:": "<class 'dict'>", ":serialized:": "gAWV", "activation_fn": "<class 'torch.nn.modules.activation.ELU'>"}
    with pytest.raises(ValueError, match="ReLU and Tanh"):
        load_sb3_checkpoint(write_zip(tmp_path / "elu.zip", sd, pk))
    with pytest.raises(ValueError, match="relu"):
        load_sb3_checkpoint(sd, activation="elu")


def test_zip_is_never_unpickled(tmp_path):
    """a zip whose policy.pth holds a pickled object that is not a tensor is refused by weights_only loading"""
    buf = io.BytesIO()
    torch.save({"x": torch.zeros(2), "obj": _Unsafe()}, buf)
    with zipfile.ZipFile(tmp_path / "bad.zip", "w") as z:
        z.writestr("policy.pth", buf.getvalue())
    with pytest.raises(Exception) as e:
        load_sb3_checkpoint(tmp_path / "bad.zip")
    assert not isinstance(e.value, _Unsafe.Ran)


class _Unsafe:
    class Ran(Exception):
        pass

    def __reduce__(self):
        return (_unsafe_called, ())


def _unsafe_called():
    raise _Unsafe.Ran("unpickled")


def _drop(sd, *prefixes):
    return {k: v for k, v in sd.items() if not k.startswith(prefixes)}


REJECTIONS = [
    ("gSDE SAC", lambda: {**_drop(sp.sac_state_dict(0, widths=(32,)), "actor.log_std"),
                          "actor.log_std": np.zeros((32, 2), np.float32)}, "gSDE"),
    ("gSDE SAC mu", lambda: {**{("actor.mu.0." + k.split(".")[-1] if k.startswith("actor.mu.") else k): v
                                for k, v in sp.sac_state_dict(0, widths=(32,)).items()}}, "gSDE"),
    ("gSDE PPO", lambda: {**sp.ppo_state_dict(0, widths=(32,)), "log_std": np.zeros((32, 2), np.float32)}, "gSDE"),
    ("feature extractor", lambda: {**sp.ppo_state_dict(0, widths=(32,)),
                                   "features_extractor.cnn.0.weight": np.zeros((4, 1, 3, 3), np.float32)}, "feature extractor"),
    ("TD3", lambda: {"actor.mu.0.weight": np.zeros((32, 1080), np.float32), "actor.mu.0.bias": np.zeros(32, np.float32),
                     "actor_target.mu.0.weight": np.zeros((32, 1080), np.float32)}, "TD3"),
    ("missing SAC head", lambda: _drop(sp.sac_state_dict(0, widths=(32,)), "actor.log_std"), "missing"),
    ("missing PPO head", lambda: _drop(sp.ppo_state_dict(0, widths=(32,)), "action_net"), "missing"),
    ("missing PPO log_std", lambda: _drop(sp.ppo_state_dict(0, widths=(32,)), "log_std"), "missing"),
    ("five layers", lambda: sp.sac_state_dict(0, widths=(16,) * 5), "at most 4"),
    ("too wide", lambda: sp.ppo_state_dict(0, widths=(1028,)), "1024"),
    ("no hidden layer", lambda: _drop(sp.ppo_state_dict(0, widths=(32,)), "mlp_extractor.policy_net"), "hidden layer"),
    ("unknown", lambda: {"q_net.0.weight": np.zeros((2, 2), np.float32)}, "not an SB3"),
]


@pytest.mark.parametrize("name,make,match", REJECTIONS, ids=[r[0] for r in REJECTIONS])
def test_rejections(name, make, match):
    with pytest.raises(ValueError, match=match):
        load_sb3_checkpoint(make(), n_beams=1080)


def test_first_layer_must_read_n_beams():
    sd = sp.sac_state_dict(0, n_beams=540, widths=(32,))
    assert load_sb3_checkpoint(sd, n_beams=540)[2]["in_features"] == 540
    with pytest.raises(ValueError, match="1080 beams"):
        load_sb3_checkpoint(sd, n_beams=1080)


def torch_actor(sd, algo, activation, obs, eps=None, deterministic=True, shared=0):
    """the actor as torch.nn modules built from the same state dict, in float64"""
    act = {"relu": torch.nn.ReLU, "tanh": torch.nn.Tanh}[activation]
    w = {k: torch.as_tensor(v, dtype=torch.float64) for k, v in sd.items()}

    def seq(prefix):
        idx = sorted({int(m.group(1)) for k in w for m in [re.fullmatch(re.escape(prefix) + r"\.(\d+)\.weight", k)] if m})
        mods = []
        for i in idx:
            lin = torch.nn.Linear(w[f"{prefix}.{i}.weight"].shape[1], w[f"{prefix}.{i}.weight"].shape[0]).double()
            lin.load_state_dict({"weight": w[f"{prefix}.{i}.weight"], "bias": w[f"{prefix}.{i}.bias"]})
            mods += [lin, act()]
        return torch.nn.Sequential(*mods)

    def lin(prefix):
        m = torch.nn.Linear(w[prefix + ".weight"].shape[1], w[prefix + ".weight"].shape[0]).double()
        m.load_state_dict({"weight": w[prefix + ".weight"], "bias": w[prefix + ".bias"]})
        return m

    x = torch.as_tensor(obs, dtype=torch.float64)
    with torch.no_grad():
        if algo == "sac":
            lat = seq("actor.latent_pi")(x)
            mean, log_std = lin("actor.mu")(lat), torch.clamp(lin("actor.log_std")(lat), -20, 2)
        else:
            lat = seq("mlp_extractor.policy_net")(seq("mlp_extractor.shared_net")(x))
            mean = lin("action_net")(lat)
            log_std = w["log_std"].expand_as(mean)
        std = torch.exp(log_std)
        u = mean if deterministic else mean + std * torch.as_tensor(eps, dtype=torch.float64)
        a = torch.tanh(u) if algo == "sac" else u
    return mean.numpy(), std.numpy(), a.numpy()


@pytest.mark.parametrize("algo,kw", CASES)
@pytest.mark.parametrize("activation", ["relu", "tanh"])
def test_restatement_equals_torch(algo, kw, activation):
    sd = make_sd(algo, 4, **kw)
    _, w, _ = load_sb3_checkpoint(sd, activation=activation)
    rng = np.random.default_rng(5)
    obs = rng.uniform(0, 1, (9, 1080))
    eps = rng.standard_normal((9, 2))
    for det in (True, False):
        got = sp.actor(w, algo, activation, obs, eps, deterministic=det)
        want = torch_actor(sd, algo, activation, obs, eps, deterministic=det)
        for g, t in zip(got, want):
            np.testing.assert_allclose(g, t, rtol=1e-12, atol=1e-12)


def test_sac_log_std_clamp_and_ppo_unclipped():
    sd = sp.sac_state_dict(6, widths=(16,), log_std_bias=40.0)
    _, w, _ = load_sb3_checkpoint(sd)
    _, std, _ = sp.actor(w, "sac", "relu", np.ones((3, 1080)) * 0.5)
    np.testing.assert_allclose(std, np.exp(2.0))
    sd = sp.ppo_state_dict(6, widths=(16,), log_std=(3.0, 3.0))
    _, w, _ = load_sb3_checkpoint(sd)
    _, _, a = sp.actor(w, "ppo", "tanh", np.ones((64, 1080)) * 0.5, np.full((64, 2), 3.0), deterministic=False)
    assert np.abs(a).max() > 1.0   # the rollout buffer's action is not clipped


def test_random_action_law():
    """values 2 (x >> 8) 2^-24 - 1: exact float32 multiples of 2^-23 in [-1, 1), uniform"""
    a = random_actions(0x1234_5678_9ABC, 50000, 7)
    assert a.dtype == np.float32 and a.min() >= -1.0 and a.max() < 1.0
    assert np.all(np.float64(a) * 2 ** 23 == np.round(np.float64(a) * 2 ** 23))
    assert abs(a.mean()) < 0.01 and abs(a.var() - 1 / 3) < 0.01
    seed = 0x1234_5678_9ABC
    x = philox4x32_10(np.arange(4), 7, 0, STREAM_RANDOM, seed & 0xFFFFFFFF, (seed >> 32) ^ STREAM_RANDOM)
    np.testing.assert_array_equal(a[:4, 1], (2.0 * (x[1] >> 8) / 2.0 ** 24 - 1.0).astype(np.float32))
    assert not np.array_equal(random_actions(seed, 8, 7), random_actions(seed, 8, 8))
    np.testing.assert_array_equal(random_actions(seed, 8, 7, gid0=4)[:4], random_actions(seed, 8, 7)[4:])


def test_mlp_normals_layout():
    seed = 99
    e = mlp_normals(seed, 20000, 3)
    z = normal4(seed, np.arange(20000), 3, 0, STREAM_MLP)
    np.testing.assert_array_equal(e, z[:, :2])
    assert abs(e.mean()) < 0.03 and abs(e.std() - 1) < 0.03
    assert not np.allclose(e, normal4(seed, np.arange(20000), 3, 0, 0x5452414E)[:, :2])


def test_stream_tags_distinct():
    src = "".join((ROOT / "racing_dreamer_b200" / "csrc" / f).read_text() for f in ("rd_common.cuh", "rd_gemm.cuh"))
    tags = dict(re.findall(r"#define (RD_STREAM_\w+) (0x[0-9a-fA-F]+)u", src))
    assert {"RD_STREAM_MLP", "RD_STREAM_RANDOM", "RD_STREAM_STOCH", "RD_STREAM_ACTOR", "RD_STREAM_TRAIN",
            "RD_STREAM_LIDAR", "RD_STREAM_RESET", "RD_STREAM_STORE"} <= set(tags)
    assert len(set(int(v, 16) for v in tags.values())) == len(tags)
    assert int(tags["RD_STREAM_MLP"], 16) == STREAM_MLP and int(tags["RD_STREAM_RANDOM"], 16) == STREAM_RANDOM


NEW_SYMBOLS = ("rd_policy_mlp_init", "rd_policy_mlp", "rd_policy_mlp_set_weights", "rd_rollout_mlp", "rd_policy_random",
               "rd_rollout_random")


def test_new_abi_declared_and_bound():
    header = (ROOT / "include" / "rd_env.h").read_text()
    lib = _abi.load_library()
    for name in NEW_SYMBOLS:
        assert re.search(rf"\bint {name}\(", header), name
        assert name in _abi.EXPORTS and hasattr(lib, name)
        assert getattr(lib, name).restype is C.c_int32 and getattr(lib, name).argtypes
    for name, value in (("RD_STORE_POLICY_MLP", 3), ("RD_STORE_POLICY_MLP_TRAIN", 4), ("RD_STORE_POLICY_RANDOM", 5),
                        ("RD_ACT_RELU", 0), ("RD_ACT_TANH", 1), ("RD_HEAD_SQUASHED", 0), ("RD_HEAD_DIAG", 1)):
        assert re.search(rf"\b{name} = {value}\b", header), name
    assert (_abi.STORE_POLICY_MLP, _abi.STORE_POLICY_MLP_TRAIN, _abi.STORE_POLICY_RANDOM) == (3, 4, 5)
    for name, value in (("RD_MLP_MAX_LAYERS", 4), ("RD_MLP_MAX_WIDTH", 1024), ("RD_MLP_DEBUG_FLOATS", 4)):
        assert f"#define {name} {value}" in header and getattr(_abi, name) == value
    # rd_mlp_actor: 2 + 4 + 2 int32, 2 floats, 4 + 4 + 5 pointers
    assert C.sizeof(_abi.RdMlpActor) == 4 * 8 + 8 + 8 * 13
    assert lib.rd_policy_mlp_init(None, C.byref(_abi.RdMlpActor())) != 0
    assert lib.rd_policy_random(None, None, None) != 0


def test_baselines_config_is_the_chain():
    from racing_dreamer_b200.compat import baselines_config
    ec = baselines_config("austria", 64)
    assert (ec.n_envs, ec.normalize_obs, ec.obs_type, ec.clip_actions, ec.rescale_actions, ec.repeat_semantics,
            ec.time_limit_ticks, ec.time_limit_steps, ec.reset_mode, ec.action_repeat) == (
        64, "baselines", "lidar", True, False, "baselines", 2000, 0, "random", 4)
    t = baselines_config(["austria", "columbia"], 8, action_repeat=2, mode="test", seed=5)
    assert (t.tracks, t.time_limit_ticks, t.reset_mode, t.action_repeat, t.seed) == (("austria", "columbia"), 4000, "grid", 2, 5)
    with pytest.raises(ValueError):
        baselines_config("austria", 1, mode="eval")
