"""CPU: the 'lidar_occupancy' Dreamer agent's definition and host side -- the float64 ConvEncoder restatement
(tests/occupancy_reference.conv_encoder, [UPSTREAM-RECALL: Dreamer models.py ConvEncoder]) against torch's conv2d, which
pins the kernel layout (Keras [kh][kw][Cin][Cout]) and the (y, x, c) flatten order; the C ABI's new entry points; and
the weight-dict validation DreamerPolicy does before any device work."""
import ctypes as C

import numpy as np
import pytest
import torch

import occupancy_reference as occref
from oracle import dreamer_policy as dp
from racing_dreamer_b200 import _abi
from racing_dreamer_b200.policy import _dreamer_arch, _encoder_depth

NEW_SYMBOLS = ("rd_policy_dreamer_init_occupancy", "rd_policy_dreamer_occupancy", "rd_policy_dreamer_occupancy_train",
               "rd_policy_dreamer_set_weights_occupancy", "rd_dreamer_encode_occupancy")


def torch_encoder(w, occ):
    """the same ConvEncoder through torch.nn.functional.conv2d: NHWC -> NCHW, HWIO -> OIHW, output back to (y, x, c)"""
    x = torch.from_numpy(np.asarray(occ, np.float64)).reshape(len(occ), 64, 64, 1).permute(0, 3, 1, 2)
    for l in range(1, 5):
        k = torch.from_numpy(w[f"enc{l}_w"].astype(np.float64)).permute(3, 2, 0, 1)
        b = torch.from_numpy(w[f"enc{l}_b"].astype(np.float64))
        x = torch.relu(torch.nn.functional.conv2d(x, k, b, stride=2))
    assert tuple(x.shape[1:]) == (256, 2, 2)
    return x.permute(0, 2, 3, 1).reshape(len(occ), -1).numpy()


@pytest.mark.parametrize("kind", ["bernoulli", "zeros", "ones", "sparse"])
def test_oracle_encoder_matches_torch_conv2d(kind):
    rng = np.random.RandomState(7)
    w = occref.random_weights(3)
    n = 6
    occ = {"bernoulli": rng.rand(n, 64, 64, 1) < 0.5, "zeros": np.zeros((n, 64, 64, 1)), "ones": np.ones((n, 64, 64, 1)),
           "sparse": rng.rand(n, 64, 64, 1) < 0.05}[kind].astype(np.uint8)
    got = occref.conv_encoder(w, occ, np.float64)
    want = torch_encoder(w, occ)
    assert got.shape == (n, 1024) and got.dtype == np.float64
    assert np.abs(got - want).max() <= 1e-12 * max(1.0, np.abs(want).max())
    assert np.abs(want).max() > 0.1   # the random encoder keeps a usable scale through the ReLU stack


def test_oracle_flatten_order_and_layout():
    """one non-zero kernel tap per layer: the embed element it lands on follows (y, x, c) and [kh][kw][Cin][Cout]"""
    w = occref.random_weights(3)
    for l in range(1, 5):
        w[f"enc{l}_w"][:] = 0
        w[f"enc{l}_b"][:] = 0
    occ = np.zeros((1, 64, 64, 1), np.uint8)
    occ[0, 0, 0, 0] = 1
    w["enc1_w"][0, 0, 0, 5] = 1.0      # conv1 channel 5 at (0, 0) sees pixel (0, 0)
    w["enc2_w"][0, 0, 5, 9] = 1.0      # -> conv2 channel 9 at (0, 0)
    w["enc3_w"][0, 0, 9, 17] = 1.0     # -> conv3 channel 17 at (0, 0)
    w["enc4_w"][0, 0, 17, 200] = 2.0   # -> conv4 channel 200 at (0, 0) only
    w["enc4_b"][3] = 0.5               # and channel 3 everywhere
    e = occref.conv_encoder(w, occ)[0]
    want = np.zeros(1024)
    want[200] = 2.0
    want[[3, 256 + 3, 512 + 3, 768 + 3]] = 0.5
    np.testing.assert_array_equal(e, want)
    np.testing.assert_array_equal(torch_encoder(w, occ)[0], want)


def test_random_weights_with_encoder():
    c = occref.random_weights(9)
    assert c["obs1_w"].shape == (dp.DETER + 1024, dp.HIDDEN)
    assert [c[f"enc{l}_w"].shape for l in range(1, 5)] == [(4, 4, 1, 32), (4, 4, 32, 64), (4, 4, 64, 128), (4, 4, 128, 256)]
    # the encoder comes from a generator of its own: the other arrays are the lidar agent's draws at embed 1024
    d = dp.random_weights(9, n_beams=1024)
    assert set(c) == set(d) | set(occref.ENC_KEYS) and all(np.array_equal(c[k], d[k]) for k in d)


def test_abi_declares_and_binds_the_new_entry_points():
    lib = _abi.load_library()
    assert _abi.ABI_VERSION == 3 and lib.rd_abi_version() == 3
    for name in NEW_SYMBOLS:
        assert name in _abi.EXPORTS and hasattr(lib, name)
        assert getattr(lib, name).restype is C.c_int32 and getattr(lib, name).argtypes
    assert [f[0] for f in _abi.RdDreamerConvEncoder._fields_] == ["depth", "w", "b"]
    assert C.sizeof(_abi.RdDreamerConvEncoder) == 8 + 8 * 8


def test_init_without_a_device_fails_cleanly():
    """rd_policy_dreamer_init_occupancy with a null handle or encoder returns RD_ERR_INVALID without touching memory"""
    lib = _abi.load_library()
    s, e = _abi.RdDreamerWeights(), _abi.RdDreamerConvEncoder()
    assert lib.rd_policy_dreamer_init_occupancy(None, C.byref(s), C.byref(e)) != 0
    assert lib.rd_dreamer_encode_occupancy(None, None, None, None) != 0


def _arch_and_depth(w):
    deter, _, _, embed, _, _ = _dreamer_arch(w)
    return _encoder_depth(w, deter, embed)


def test_weight_dict_validation():
    w = occref.random_weights(5)
    assert _arch_and_depth(w) == 32
    assert _arch_and_depth(dp.random_weights(5)) == 0
    for k in ("enc1_w", "enc3_b", "enc4_w"):
        bad = dict(w)
        del bad[k]
        with pytest.raises(ValueError, match="missing"):
            _arch_and_depth(bad)
    bad = dict(w, enc2_w=np.zeros((4, 4, 32, 32), np.float32))
    with pytest.raises(ValueError, match="enc2_w has shape"):
        _arch_and_depth(bad)
    bad = dict(w, enc4_b=np.zeros(128, np.float32))
    with pytest.raises(ValueError, match="enc4_b has shape"):
        _arch_and_depth(bad)
    bad = dict(w, enc1_w=np.zeros((3, 3, 1, 32), np.float32))
    with pytest.raises(ValueError, match="enc1_w has shape"):
        _arch_and_depth(bad)
    bad = dict(w, obs1_w=np.zeros((dp.DETER + 1080, dp.HIDDEN), np.float32))
    with pytest.raises(ValueError, match="deter \\+ 32 \\* depth"):
        _arch_and_depth(bad)
    # a depth-16 encoder is a consistent dict (the C ABI, which takes depth 32 only, rejects it)
    assert _arch_and_depth(occref.random_weights(5, conv_depth=16)) == 16


def test_conv_agent_needs_an_occupancy_env(monkeypatch):
    """DreamerPolicy refuses an encoder agent on a lidar-only env before it creates anything on the device"""
    from racing_dreamer_b200.policy import DreamerPolicy

    class LidarOnlyEnv:
        n, n_beams, device = 4, 1080, "cpu"
        cfg = _abi.RdConfig()
        cfg.obs_flags = _abi.OBS_LIDAR

    with pytest.raises(ValueError, match="obs_type='lidar_occupancy'"):
        DreamerPolicy(LidarOnlyEnv(), occref.random_weights(5))
