"""CPU: the training-mode Dreamer agent step (rd_policy_dreamer_train, csrc/rd_gemm.cuh k_actor_train) restated in NumPy.

* ``ref_exploration_amount`` / ``sample`` / ``explore`` / ``train_step`` below restate Dreamer.policy(training=True) in
  float64 on top of the oracle's RSSM and actor head (oracle/dreamer_policy.py); the GPU tests compare the kernels with
  them.  The reference tree is not vendored: Dreamer.policy and _exploration are [UPSTREAM-RECALL].
* The exploration schedule of the product (policy.exploration_amount, what the library computes per step) against that
  restatement, and the env-step accounting of mixed training / evaluation steps, single- and multi-car.
* The Philox layout of the training draws: counter (env id, step, 0, RD_STREAM_TRAIN), key (seed_lo, seed_hi ^ tag),
  through the NumPy Philox that test_cpu_episode_store checks against the oracle's philox4x32_10.  ``train_normals``
  and ``posterior_normals`` are what the GPU tests feed the explicit-noise path with.
* The oracle's training step against an independent evaluation of tanh(mean + sd e1), its log-probability and the clip.
* The new C entry points are declared, exported and bound."""
import re
from pathlib import Path

import numpy as np
import pytest

from oracle import dreamer_policy as dp
from racing_dreamer_b200 import _abi
from racing_dreamer_b200.policy import env_steps_per_training_step, exploration_amount
from test_cpu_episode_store import philox4x32_10

ROOT = Path(__file__).resolve().parents[1]
STREAM_TRAIN = 0x5452414E   # RD_STREAM_TRAIN
STREAM_STOCH = 0x53544F43   # RD_STREAM_STOCH
STREAM_ACTOR = 0x41435452   # RD_STREAM_ACTOR


# Dreamer.policy(obs, state, training=True) [REF dreamer/dreamer.py, Dreamer.policy and _exploration; UPSTREAM-RECALL]:
# action = actor(feat).sample(); action = clip(Normal(action, amount).sample(), -1, 1) with amount = expl_amount *
# 0.5 ** (step / expl_decay) if expl_decay, max(expl_min, amount) if expl_min; the explored action is kept in `state`.
def ref_exploration_amount(step, expl_amount=0.3, expl_decay=0.0, expl_min=0.0):
    """Dreamer._exploration's amount at env step `step` (float64); defaults: define_config's [UPSTREAM-RECALL]."""
    amount = expl_amount
    if expl_decay:
        amount *= 0.5 ** (step / expl_decay)
    if expl_min:
        amount = max(expl_min, amount)
    return amount


def sample(mean, std, eps_sample):
    """One draw of the actor distribution, tanh(mean + std * eps), and its log_prob; eps_sample [..., 2]."""
    u, lp = dp.sample_log_prob(mean, std, eps_sample.astype(mean.dtype)[..., None, :])
    return np.tanh(u[..., 0, :]), lp[..., 0]


def explore(action, amount, eps_expl):
    """Normal(action, amount).sample() with the standard-normal draw eps_expl, clipped to [-1, 1]."""
    return np.clip(action + amount * eps_expl.astype(action.dtype), -1.0, 1.0)


def train_step(w, scan, state, eps_stoch, eps_sample, eps_expl, amount, dtype=np.float64):
    """Dreamer.policy(training=True) for a batch: (explored action, new state, diagnostics)."""
    n = scan.shape[0]
    embed = dp.preprocess_lidar(scan)
    if state is None:
        stoch, deter, action = np.zeros((n, dp.STOCH), dtype), np.zeros((n, dp.DETER), dtype), np.zeros((n, 2), dtype)
    else:
        stoch, deter, action = state
    mean, std, stoch, deter = dp.obs_step(w, stoch, deter, action, embed, eps_stoch, dtype)
    feat = np.concatenate([stoch, deter], -1)
    amean, astd = dp.actor_dist(w, feat, dtype)
    a, logp = sample(amean, astd, eps_sample)
    act = explore(a, amount, eps_expl)
    return act, (stoch, deter, act), dict(mean=mean, std=std, actor_mean=amean, actor_std=astd, sample=a, logp=logp)


def normal4(seed, gid, step, c2, tag):
    """gm_normal4 in float64: Philox4x32-10(counter (gid, step, c2, tag), key (seed_lo, seed_hi ^ tag)), Box-Muller on
    u1 = ((x >> 8) + 1) / 2^24 in (0, 1] and u2 = (x >> 8) / 2^24 in [0, 1) -> [..., 4]."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    x = philox4x32_10(gid, step, c2, tag, seed & 0xFFFFFFFF, (seed >> 32) ^ tag)
    z = []
    for h in range(2):
        u1 = ((x[2 * h] >> 8).astype(np.float64) + 1.0) / 16777216.0
        u2 = (x[2 * h + 1] >> 8).astype(np.float64) / 16777216.0
        r = np.sqrt(-2.0 * np.log(u1))
        z += [r * np.cos(2.0 * np.pi * u2), r * np.sin(2.0 * np.pi * u2)]
    return np.stack(z, -1)


def train_normals(seed, n, step, gid0=0):
    """(e1 [n,2], e2 [n,2]) of training step `step`: the sample's and the exploration's standard normals."""
    z = normal4(seed, np.arange(n) + gid0, step, 0, STREAM_TRAIN)
    return z[:, :2], z[:, 2:]


def posterior_normals(seed, n, step, gid0=0):
    """eps_stoch [n,30] of the posterior sample at agent step `step`: latent j from block (gid, step, 4 (j // 4), tag)."""
    return np.concatenate([normal4(seed, np.arange(n) + gid0, step, j0, STREAM_STOCH) for j0 in range(0, 32, 4)], -1)[:, :30]


@pytest.mark.parametrize("amount,decay,floor", [(0.3, 0.0, 0.0), (0.3, 5e5, 0.0), (0.3, 5e5, 0.05), (0.3, 0.0, 0.5),
                                                (1.0, 1234.5, 0.0), (0.0, 0.0, 0.1)])
def test_schedule_equals_the_restated_formula(amount, decay, floor):
    for step in [0, 1, 8, 4096 * 8, 123457, 5 * 10 ** 5, 2 * 10 ** 6, 10 ** 8]:
        want = np.float32(ref_exploration_amount(step, amount, decay, floor))
        got = exploration_amount(amount, decay, floor, step)
        assert got.dtype == np.float32 and got == want, (step, got, want)
    if decay == 0.0:   # no decay: constant, floored
        assert exploration_amount(amount, decay, floor, 10 ** 9) == np.float32(max(amount, floor))
    else:              # halves every `decay` env steps until the floor
        a0, a1 = exploration_amount(amount, decay, 0.0, 0), exploration_amount(amount, decay, 0.0, 2 * decay)
        assert abs(float(a1) - float(a0) / 4) <= 1e-7 * float(a0)


@pytest.mark.parametrize("n_envs,repeat,agents", [(4096, 8, 1), (16, 4, 1), (12, 4, 3)])
def test_env_steps_accounting(n_envs, repeat, agents):
    """Dreamer's step counter: + len(reset) * action_repeat per training call (one entry per car), eval calls leave it;
    the amount of each training step is the schedule at the counter BEFORE that step's increment."""
    cfg = _abi.RdConfig()
    cfg.n_envs, cfg.action_repeat, cfg.agents_per_world = n_envs, repeat, agents
    per = env_steps_per_training_step(cfg)
    assert per == n_envs * repeat
    kinds = ["train", "train", "eval", "train", "eval", "eval", "train"]
    steps, ref_step, amounts, ref_amounts = 0, 0, [], []
    for k in kinds:
        if k == "train":
            amounts.append(exploration_amount(0.3, 5 * per, 0.1, steps))
            steps += per
            ref_amounts.append(np.float32(ref_exploration_amount(ref_step, 0.3, 5 * per, 0.1)))
            ref_step += n_envs * repeat   # self._step.assign_add(len(reset) * action_repeat)
    assert steps == ref_step == kinds.count("train") * n_envs * repeat
    assert amounts == ref_amounts and amounts[0] == np.float32(0.3) and amounts[1] < amounts[0]


def test_stream_tag_and_layout():
    src = (ROOT / "racing_dreamer_b200" / "csrc" / "rd_gemm.cuh").read_text()
    tags = {n: int(v, 16) for n, v in re.findall(r"#define (RD_STREAM_\w+) 0x([0-9a-fA-F]+)u", src)}
    assert tags["RD_STREAM_TRAIN"] == STREAM_TRAIN and tags["RD_STREAM_STOCH"] == STREAM_STOCH
    common = (ROOT / "racing_dreamer_b200" / "csrc" / "rd_common.cuh").read_text()
    tags.update({n: int(v, 16) for n, v in re.findall(r"#define (RD_STREAM_\w+) 0x([0-9a-fA-F]+)u", common)})
    assert len(set(tags.values())) == len(tags), "every Philox stream has its own tag"
    assert re.search(r"gm_normal4\(g\.gid0 \+ \(uint32_t\)row, g\.step, 0u, RD_STREAM_TRAIN, g\.key0, g\.key1, z\)", src)
    assert "(uint32_t)(seed >> 32) ^ RD_STREAM_TRAIN" in (ROOT / "racing_dreamer_b200" / "csrc" / "rd_dreamer.cuh").read_text()


def test_training_draws_on_the_numpy_philox():
    seed = 0x0123456789ABCDEF
    e1, e2 = train_normals(seed, 8, 5, gid0=100)
    # the same block as a direct Philox call: counter (gid, step, 0, tag), key (seed_lo, seed_hi ^ tag)
    x = philox4x32_10(np.array([103]), 5, 0, STREAM_TRAIN, seed & 0xFFFFFFFF, (seed >> 32) ^ STREAM_TRAIN)
    u1, u2 = ((int(x[0][0]) >> 8) + 1) / 2 ** 24, (int(x[1][0]) >> 8) / 2 ** 24
    assert e1[3, 0] == np.sqrt(-2 * np.log(u1)) * np.cos(2 * np.pi * u2)
    # independent of the evaluation-mode actor stream and of the posterior stream at the same (env, step)
    ea = normal4(seed, np.arange(8) + 100, 5, 0, STREAM_ACTOR)
    es = posterior_normals(seed, 8, 5, gid0=100)
    assert not np.allclose(ea[:, :2], e1) and not np.allclose(es[:, :2], e1)
    # per env, per step and per rank (env_id_offset) different; the same for the same (seed, env, step)
    assert not np.allclose(train_normals(seed, 8, 6, 100)[0], e1) and not np.allclose(train_normals(seed, 8, 5, 0)[0], e1)
    assert np.array_equal(train_normals(seed, 8, 5, 100)[1], e2)
    z = np.concatenate([np.concatenate(train_normals(7, 4096, s), -1) for s in range(8)]).ravel()
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01


def test_training_step_restatement_against_an_independent_evaluation():
    rng = np.random.RandomState(2)
    w = dp.random_weights(3, n_beams=64)
    n = 64
    scan = rng.uniform(0, 20, (n, 64))
    state = (rng.standard_normal((n, 30)), rng.uniform(-1, 1, (n, 200)), rng.uniform(-1, 1, (n, 2)))
    es, e1, e2 = rng.standard_normal((n, 30)), rng.standard_normal((n, 2)), rng.standard_normal((n, 2))
    amount = 0.3
    act, new_state, d = train_step(w, scan, state, es, e1, e2, amount)
    # the mode step's RSSM and actor distribution are shared
    _, mstate, md = dp.policy_step(w, scan, state, es, rng.standard_normal((n, 4, 2)))
    assert np.array_equal(mstate[1], new_state[1]) and np.array_equal(md["actor_mean"], d["actor_mean"])
    mean, std = d["actor_mean"], d["actor_std"]
    u = mean + std * e1
    a = np.tanh(u)
    assert np.allclose(d["sample"], a, rtol=0, atol=1e-15)
    # log N(u; mean, std) - log|d tanh(u)/du| per dimension, summed
    logn = -0.5 * ((u - mean) / std) ** 2 - np.log(std) - 0.5 * np.log(2 * np.pi)
    logdet = np.log(1.0 - np.tanh(u) ** 2)
    ok = np.abs(u) < 5   # 1 - tanh^2 loses its digits beyond that; the oracle's form does not
    assert np.allclose((logn - logdet).sum(-1)[ok.all(-1)], d["logp"][ok.all(-1)], rtol=1e-9, atol=1e-9)
    want = np.minimum(np.maximum(a + amount * e2, -1.0), 1.0)
    assert np.array_equal(act, want) and np.array_equal(new_state[2], act)
    assert ((act == 1.0) | (act == -1.0)).any() and (np.abs(act) < 1).any()
    # zero draws: tanh(mean), what the evaluation step with zero noise gives
    z = np.zeros((n, 2))
    act0, _, _ = train_step(w, scan, state, es, z, z, amount)
    m0, _, _, _ = dp.mode(mean, std, None)
    assert np.array_equal(act0, m0)


def test_new_symbols_declared_and_bound():
    header = (ROOT / "include" / "rd_env.h").read_text()
    for name in ("rd_policy_dreamer_set_exploration", "rd_policy_dreamer_get_exploration", "rd_policy_dreamer_train",
                 "rd_rollout_dreamer_train", "rd_policy_dreamer_set_weights"):
        assert re.search(rf"\bint {name}\(", header), name
        assert name in _abi.EXPORTS
        assert getattr(_abi.load_library(), name).restype is not None
    assert "RD_STORE_POLICY_DREAMER_TRAIN = 2" in header and _abi.STORE_POLICY_DREAMER_TRAIN == 2
    assert [f for f, _ in _abi.RdDreamerExploration._fields_] == ["amount", "decay", "min_amount", "env_steps"]
    assert _abi.ABI_VERSION == 3 and "#define RD_ABI_VERSION 3" in header
