"""CPU: DreamerAgents' host-side rejections, made before any device work (the env below has no library)."""
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import dreamer_policy as dp
from racing_dreamer_b200 import _abi
from racing_dreamer_b200.policy import DreamerAgents


class NoDeviceEnv(SimpleNamespace):
    """Only what DreamerAgents validates against; any library call fails the test."""

    @property
    def lib(self):
        raise AssertionError("DreamerAgents reached the device before rejecting its arguments")


@pytest.fixture(scope="module")
def env():
    return NoDeviceEnv(n=8, n_beams=1080, cfg=SimpleNamespace(obs_flags=0), device="cpu")


@pytest.fixture(scope="module")
def w():
    return [dp.random_weights(41), dp.random_weights(42, normalized=True)]


def test_architecture_mismatch(env, w):
    with pytest.raises(ValueError, match="checkpoint 1 does not match checkpoint 0's architecture: deter 100 != 200"):
        DreamerAgents(env, [w[0], dp.random_weights(43, deter=100)], np.arange(8) % 2)
    with pytest.raises(ValueError, match="units 64 != 400"):
        DreamerAgents(env, [w[0], dp.random_weights(43, units=64)], np.arange(8) % 2)
    # a single checkpoint's own defects keep _dreamer_arch's message
    bad = dict(w[1])
    del bad["obs2_b"]
    with pytest.raises(ValueError, match="checkpoint array obs2_b is missing"):
        DreamerAgents(env, [w[0], bad], np.arange(8) % 2)
    with pytest.raises(ValueError, match="the checkpoint embeds 512 beams, the env casts 1080"):
        DreamerAgents(env, [dp.random_weights(1, n_beams=512)] * 2, np.arange(8) % 2)


def test_agent_ids(env, w):
    with pytest.raises(ValueError, match=r"values must be in \[0, 2\)"):
        DreamerAgents(env, w, np.array([0, 1, 2, 0, 1, 0, 1, 0]))
    with pytest.raises(ValueError, match=r"values must be in \[0, 2\)"):
        DreamerAgents(env, w, np.array([0, 1, -1, 0, 1, 0, 1, 0]))
    with pytest.raises(ValueError, match=r"agents \[1\] drive no env"):
        DreamerAgents(env, w, np.zeros(8, np.int32))


def test_agent_count(env, w):
    many = [w[0]] * (_abi.RD_MAX_DREAMER_AGENTS + 1)
    with pytest.raises(ValueError, match="9 checkpoints: expected 1..8 agents"):
        DreamerAgents(env, many, np.arange(8) % 8)
    with pytest.raises(ValueError, match="0 checkpoints"):
        DreamerAgents(env, [], np.zeros(8, np.int32))
    with pytest.raises(TypeError, match="sequence"):
        DreamerAgents(env, w[0], np.zeros(8, np.int32))


def test_agent_of_env_shape_and_dtype(env, w):
    with pytest.raises(ValueError, match=r"shape \(8,\)"):
        DreamerAgents(env, w, np.arange(7) % 2)
    with pytest.raises(ValueError, match=r"shape \(8,\)"):
        DreamerAgents(env, w, (np.arange(8) % 2).reshape(2, 4))
    with pytest.raises(ValueError, match="integer array"):
        DreamerAgents(env, w, (np.arange(8) % 2).astype(np.float32))


def test_per_agent_exploration_and_options(env, w):
    with pytest.raises(ValueError, match=r"expl_amount: one value, or one per agent \(2\)"):
        DreamerAgents(env, w, np.arange(8) % 2, expl_amount=[0.3, 0.2, 0.1])
    with pytest.raises(ValueError, match="noise"):
        DreamerAgents(env, w, np.arange(8) % 2, noise="gaussian")
    with pytest.raises(ValueError, match="precision"):
        DreamerAgents(env, w, np.arange(8) % 2, precision="fp16")
