"""GPU: the 'lidar_occupancy' Dreamer agent -- the ConvEncoder (rd_gemm.cuh k_conv1, then k_dense<..., CONV> implicit
GEMMs for conv2..conv4, driven by rd_dreamer.cuh dreamer_encode) in front of the unchanged RSSM and actor -- against
the float64 restatement (tests/occupancy_reference.py over oracle/dreamer_policy.py).

Env counts.  What a batch of N envs occupies in each stage: k_conv1 one CTA per (env, output row); conv2 two 128-row
tiles per env (16 x 8 output positions each), conv3 one tile per two envs (8 x 8 positions x 2), conv4 one tile per 32
envs (2 x 2 positions x 32) -- its box runs past the last env when N is not a multiple; obs1 and everything after it
128 envs per tile.  So 1, 2, 3 (conv3's two-env tiles, odd tail), 31, 32, 33 (conv4's 32-env tiles), 127, 128, 129
(the 128-env tiles of the RSSM and actor), 300 and 4096 (many full waves).

Images: real k_occupancy images at random poses on two tracks, Bernoulli(0.5) images, all-zero and all-one images
(rows i % 4 = 0, 1, 2, 3 of a batch).

Bars: test_gpu_dreamer_shapes's error model with the encoder as a stage in front of obs1.  conv1 reads exact 0 / 1
inputs in float32 (factor 1).  tf32x3: conv2..conv4 are cut into accumulator groups as dr_build cuts obs1 (16, 32 and
64 K blocks in 3, 6 and 7 groups; the longest group 10 blocks against the shipped obs1's 6), tf32: sqrt(K / 1280) with
K up to 2048.  The embed takes the encoder's factor, the posterior and actor head the larger of it and their own.  In
tf32x3 the embed's error also stays within 8x the float32 evaluation's plus the documented floor."""
import math

import numpy as np
import pytest

import occupancy_reference as occref
from oracle import dreamer_policy as dp
from test_cpu_dreamer_train import explore, sample
from test_gpu_dreamer import BARS, check_mode, close
from test_gpu_dreamer_shapes import F32_MULTIPLE, FREE_RUNNING, _per_group, bar_factors, compare_step
from test_gpu_dreamer_train import explored

pytestmark = pytest.mark.gpu
ENVS = (1, 2, 3, 31, 32, 33, 127, 128, 129, 300, 4096)
PRECISIONS = ("tf32x3", "tf32")
DEPTH = 32
CONV_KB = (16, 32, 64)   # K blocks of conv2..conv4: 16 Cin / 32


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


def make_env(n_envs, **kw):
    from racing_dreamer_b200 import BatchedRaceEnv, EnvConfig
    base = dict(tracks=("austria", "columbia"), action_repeat=4, reset_mode="random", seed=3, obs_type="lidar_occupancy")
    base.update(kw)
    return BatchedRaceEnv(EnvConfig(n_envs=n_envs, **base), device="cuda:0")


def f32(x):
    return np.asarray(x, np.float32)


def images(torch, env, seed):
    """the env's own images at its reset poses, with rows 1, 2, 3 (mod 4) replaced by Bernoulli, all-zero, all-one"""
    env.reset()
    occ = env.buf["occupancy"].clone()
    rng = np.random.RandomState(seed)
    n = occ.shape[0]
    occ[1::4] = torch.from_numpy((rng.rand(len(range(1, n, 4)), 64, 64, 1) < 0.5).astype(np.uint8)).cuda()
    occ[2::4] = 0
    occ[3::4] = 1
    return occ


def encode_ref(w, occ, dtype=np.float64, chunk=512):
    return np.concatenate([occref.conv_encoder(w, occ[i:i + chunk], dtype) for i in range(0, len(occ), chunk)])


def enc_factor(precision):
    if precision == "tf32x3":
        shipped = _per_group(-(-200 // 32) + -(-1080 // 32), 7)
        return max(1.0, max(_per_group(kb, 7) for kb in CONV_KB) / shipped)
    return max(1.0, math.sqrt(32 * CONV_KB[-1] / (200 + 1080)))


def factors(precision):
    """[deter, posterior, actor head] bar factors: the lidar model's, with the encoder in front of obs1"""
    fac = bar_factors(200, 200, 400, 32 * DEPTH, precision)
    e = enc_factor(precision)
    return [fac[0], max(fac[1], e), max(fac[2], e)]


def random_state(rng, n):
    return f32(rng.standard_normal((n, 30))), f32(rng.uniform(-1, 1, (n, 200))), f32(rng.uniform(-1, 1, (n, 2)))


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("n", ENVS)
def test_encoder_against_float64(torch_cuda, n, precision):
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    w = occref.random_weights(200)
    env = make_env(n)
    occ = images(torch, env, n)
    pol = DreamerPolicy(env, w, precision=precision)
    got = pol.encode(occ).cpu().numpy()
    o = occ.cpu().numpy()
    want = encode_ref(w, o)
    rtol, atol, _ = BARS[precision]
    f = enc_factor(precision)
    err = close(f"embed [{precision} N{n}]", got, want, rtol * f, atol * f)
    if precision == "tf32x3":
        e32 = float(np.abs(encode_ref(w, o, np.float32).astype(np.float64) - want).max())
        assert err <= F32_MULTIPLE * e32 + atol, f"embed: {err:.3e} vs float32 evaluation {e32:.3e}"
    assert np.abs(want).max() > 0.1
    # the default input is the env's current image
    torch.cuda.synchronize()
    assert torch.equal(pol.encode(), pol.encode(env.buf["occupancy"]))
    env.close()


def _explicit(torch, pol, occ, state, es, ea):
    pol.set_state(*[torch.from_numpy(s) for s in state])
    act = pol.act(eps_stoch=torch.from_numpy(es), eps_actor=torch.from_numpy(ea), debug=True, occupancy=occ).clone()
    return act.cpu().numpy(), {k: v.cpu().numpy() for k, v in pol.diagnostics().items()}, pol.diagnostics()


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("head", ["tanh_normal", "normalized"])
def test_teacher_forced_steps(torch_cuda, head, precision):
    """evaluation step, a free-running second step, and a training step, against the oracle with explicit draws"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n, S = 300, 100
    x3 = precision == "tf32x3"
    w = occref.random_weights(300, normalized=(head == "normalized"))
    env = make_env(n)
    occ = images(torch, env, 1)
    o = occ.cpu().numpy()
    pol = DreamerPolicy(env, w, noise="explicit", n_samples=S, precision=precision)
    fac = factors(precision)
    rng = np.random.RandomState(2)

    # 1. evaluation step from a random latent state
    state = random_state(rng, n)
    es, ea = f32(rng.standard_normal((n, 30))), f32(rng.standard_normal((n, S, 2)))
    act, d, diag = _explicit(torch, pol, occ, state, es, ea)
    st, de, ac = (t.cpu().numpy() for t in pol.get_state())
    s64 = tuple(s.astype(np.float64) for s in state)
    act_ref, new_state, ref = occref.policy_step(w, o, s64, es, ea, np.float64)
    _, state32, ref32 = occref.policy_step(w, o, state, es, ea, np.float32)
    compare_step(act, d, st, de, act_ref, ref, new_state, ea, precision, fac, *((ref32, state32) if x3 else ()))
    check_mode(diag, ref, precision=precision, tie=fac[2])
    assert np.abs(ac - act).max() <= (2.0 ** -20 if x3 else 2.0 ** -11)

    # 2. free-running second step (latent kept on the device; previous action the oracle's)
    pol.set_state(action=torch.from_numpy(f32(act_ref)))
    es2, ea2 = f32(rng.standard_normal((n, 30))), f32(rng.standard_normal((n, S, 2)))
    act2 = pol.act(eps_stoch=torch.from_numpy(es2), eps_actor=torch.from_numpy(ea2), debug=True, occupancy=occ).cpu().numpy()
    diag2 = pol.diagnostics()
    d2 = {k: v.cpu().numpy() for k, v in diag2.items()}
    st2, de2, _ = (t.cpu().numpy() for t in pol.get_state())
    act_ref2, new_state2, ref2 = occref.policy_step(w, o, (new_state[0], new_state[1], f32(act_ref).astype(np.float64)), es2, ea2,
                                                np.float64)
    compare_step(act2, d2, st2, de2, act_ref2, ref2, new_state2, ea2, precision, [FREE_RUNNING * f for f in fac])
    check_mode(diag2, ref2, precision=precision, tie=FREE_RUNNING * fac[2])

    # 3. training step: one sample + exploration
    rtol, atol, hf = BARS[precision]
    state = random_state(rng, n)
    pol.set_state(*[torch.from_numpy(s) for s in state])
    es, e1, e2 = f32(rng.standard_normal((n, 30))), f32(rng.standard_normal((n, 2))), f32(rng.standard_normal((n, 2)))
    amount = pol.exploration_amount()
    act = pol.act(eps_stoch=torch.from_numpy(es), training=True, eps_sample=torch.from_numpy(e1),
                  eps_expl=torch.from_numpy(e2), debug=True, occupancy=occ).cpu().numpy()
    d = {k: v.cpu().numpy() for k, v in pol.diagnostics().items()}
    st, de, ac = (t.cpu().numpy() for t in pol.get_state())
    s64 = tuple(s.astype(np.float64) for s in state)
    mean, std, stoch, deter = dp.obs_step(w, s64[0], s64[1], s64[2], encode_ref(w, o), es, np.float64)
    amean, astd = dp.actor_dist(w, np.concatenate([stoch, deter], -1), np.float64)
    a_ref, _ = sample(amean, astd, e1)
    close("mean", d["mean"], mean, rtol * fac[1], atol * fac[1])
    close("deter", de, deter, rtol * fac[0], atol * fac[0])
    close("stoch", st, stoch, rtol * fac[1], atol * fac[1])
    close("actor_mean", d["actor_mean"], amean, rtol * hf * fac[2], atol * hf * fac[2], dp.MEAN_SCALE)
    close("actor_std", d["actor_std"], astd, rtol * hf * fac[2], atol * hf * fac[2], dp.MEAN_SCALE)
    bar = (atol + rtol * dp.MEAN_SCALE) * hf * fac[2] * (1 + np.abs(e1))
    assert (np.abs(d["action"] - a_ref) <= bar).all(), np.abs(d["action"] - a_ref).max()
    assert np.abs(explore(a_ref, float(amount), e2) - act).max() <= bar.max() + 1e-6
    assert np.array_equal(act, explored(d["action"], amount, e2))
    assert pol.env_steps == n * 4
    assert np.abs(ac - act).max() <= (2.0 ** -20 if x3 else 2.0 ** -10)
    env.close()


@pytest.mark.parametrize("training", [False, True])
def test_rollout_equals_stepwise(torch_cuda, training):
    """rd_rollout_dreamer(_train) on the env's own images == n x (act -> env.step), bit for bit, through resets"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n, steps = 300, 40
    w = occref.random_weights(500)
    outs = []
    for mode in ("rollout", "stepwise"):
        env = make_env(n, seed=6, auto_reset=True, time_limit_steps=15)
        env.reset()
        pol = DreamerPolicy(env, w, noise="philox")
        if mode == "rollout":
            pol.rollout(steps, training=training)
        else:
            for _ in range(steps):
                env.step(pol.act(training=training))
        torch.cuda.synchronize()
        outs.append((env.buf["pose"].clone(), env.buf["occupancy"].clone(), pol.actions.clone()) + tuple(pol.get_state()))
        env.close()
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def test_recorded_training_rollout_equals_loop(torch_cuda):
    """rollout(n, training=True, store=store) == act(training=True) + store.step, the store keeping lidar_occupancy"""
    torch = torch_cuda
    from racing_dreamer_b200 import BatchedRaceEnv, DreamerPolicy, EnvConfig
    from racing_dreamer_b200.episodes import DeviceEpisodeStore
    w = occref.random_weights(501)
    ec = EnvConfig(tracks=("austria", "columbia"), n_envs=16, action_repeat=4, auto_reset=False, reset_mode="random",
                   time_limit_steps=30, seed=11, obs_type="lidar_occupancy")
    runs = []
    for mode in ("rollout", "loop"):
        env = BatchedRaceEnv(ec, device="cuda:0")
        store = DeviceEpisodeStore(env, capacity_rows=400, keep_obs=("lidar", "lidar_occupancy", "pose", "speed"))
        pol = DreamerPolicy(env, w, noise="philox")
        store.reset()
        if mode == "rollout":
            pol.rollout(70, training=True, store=store)
        else:
            for _ in range(70):
                store.step(pol.act(training=True))
        torch.cuda.synchronize()
        runs.append((store.episodes(), pol.env_steps))
        env.close()
    (e1, s1), (e2, s2) = runs
    assert len(e1) == len(e2) >= 16 and s1 == s2 == 70 * 16 * 4
    assert any(np.asarray(x["lidar_occupancy"]).any() for x in e1)
    for x, y in zip(e1, e2):
        assert x.keys() == y.keys() and "lidar_occupancy" in x
        for k in x:
            assert np.array_equal(np.asarray(x[k]).view(np.uint8), np.asarray(y[k]).view(np.uint8)), k


def _outputs(torch, pol, occ, seed):
    rng = np.random.RandomState(seed)
    n = occ.shape[0]
    state = random_state(rng, n)
    es, ea = f32(rng.standard_normal((n, 30))), f32(rng.standard_normal((n, 100, 2)))
    pol.set_state(*[torch.from_numpy(s) for s in state])
    act = pol.act(eps_stoch=torch.from_numpy(es), eps_actor=torch.from_numpy(ea), debug=True, occupancy=occ).clone()
    return [pol.encode(occ), act, pol.debug.clone()] + list(pol.get_state())


def _same(torch, got, want, what):
    for j, (x, y) in enumerate(zip(got, want)):
        assert torch.equal(x, y), f"{what}: output {j} differs"


@pytest.mark.parametrize("precision", PRECISIONS)
def test_load_weights_equals_fresh_policy(torch_cuda, precision):
    """load_weights from numpy and from CUDA tensors == a policy built with those weights; a rejected refresh changes
    nothing"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 129
    w0, w1 = occref.random_weights(600), occref.random_weights(601)
    env_a, env_b = make_env(n), make_env(n)
    occ = images(torch, env_a, 3)
    fresh = _outputs(torch, DreamerPolicy(env_b, w1, noise="explicit", precision=precision), occ, 9)
    pol = DreamerPolicy(env_a, w0, noise="explicit", precision=precision)
    pol.load_weights(w1)
    _same(torch, _outputs(torch, pol, occ, 9), fresh, "numpy refresh")
    pol.load_weights(w0)
    pol.load_weights({k: torch.from_numpy(v).cuda() for k, v in w1.items()})
    _same(torch, _outputs(torch, pol, occ, 9), fresh, "CUDA refresh")
    # rejected refreshes: missing encoder array, another depth, no encoder, the lidar entry point
    bad = dict(w0)
    del bad["enc3_w"]
    w16 = occref.random_weights(602, conv_depth=16)
    lidar_w = dp.random_weights(603, n_beams=32 * DEPTH)
    for b in (bad, w16, lidar_w):
        with pytest.raises(ValueError):
            pol.load_weights(b)
    with pytest.raises(RuntimeError, match="occupancy entry points"):
        pol.env._check(pol.env.lib.rd_policy_dreamer_set_weights(pol.env._handle, None, 0, pol.env._stream()))
    _same(torch, _outputs(torch, pol, occ, 9), fresh, "after rejected refreshes")
    env_a.close()
    env_b.close()


def test_rejections_and_reinit(torch_cuda):
    """entry point / agent kind mismatches, an env without occupancy, unsupported depths; re-init both ways"""
    import ctypes as C
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy, _abi
    n = 64
    wc = occref.random_weights(700)
    wl = dp.random_weights(701)
    env = make_env(n)
    occ = images(torch, env, 4)
    lib, h, s = env.lib, env._handle, env._stream()
    pol = DreamerPolicy(env, wc)
    embed = pol.encode(occ).clone()
    act = torch.zeros((n, 2), dtype=torch.float32, device="cuda:0")
    # a conv agent refuses the lidar entry points
    with pytest.raises(RuntimeError, match="occupancy entry points"):
        env._check(lib.rd_policy_dreamer(h, env.buf["lidar"].data_ptr(), act.data_ptr(), 0, None, None, None, s))
    with pytest.raises(RuntimeError, match="occupancy entry points"):
        env._check(lib.rd_policy_dreamer_train(h, env.buf["lidar"].data_ptr(), act.data_ptr(), 0, None, None, None, None, s))
    with pytest.raises(ValueError, match="occupancy="):
        pol.act(env.buf["lidar"])
    for bad in (env.buf["occupancy"].view(n, 4096), env.buf["occupancy"].float(), env.buf["occupancy"].cpu()):
        with pytest.raises(ValueError, match="uint8"):
            pol.act(occupancy=bad)
    # a rollout without the images
    out = _abi.RdOutputs.from_buffer_copy(env._out)
    out.occupancy_dev = None
    with pytest.raises(RuntimeError, match="occupancy_dev"):
        env._check(lib.rd_rollout_dreamer(h, 1, C.byref(out), None, 1, s))
    # unsupported depth: rejected by the C ABI, the current agent keeps working
    with pytest.raises(RuntimeError, match="depth"):
        DreamerPolicy(env, occref.random_weights(702, conv_depth=16))
    assert torch.equal(pol.encode(occ), embed)
    pol.act(occupancy=occ)
    # re-init to a lidar agent: the occupancy entry points are refused, the lidar ones work
    lid = DreamerPolicy(env, wl)
    lid.act()
    with pytest.raises(RuntimeError, match="lidar entry points"):
        env._check(lib.rd_policy_dreamer_occupancy(h, occ.data_ptr(), act.data_ptr(), 0, None, None, None, s))
    with pytest.raises(RuntimeError, match="lidar entry points"):
        env._check(lib.rd_dreamer_encode_occupancy(h, occ.data_ptr(), act.data_ptr(), s))
    with pytest.raises(ValueError):
        lid.encode()
    # and back: the same encoder again
    again = DreamerPolicy(env, wc)
    assert torch.equal(again.encode(occ), embed)
    env.close()
    # an env without occupancy output: refused by the policy and by the C ABI
    lidar_env = make_env(n, obs_type="lidar")
    with pytest.raises(ValueError, match="lidar_occupancy"):
        DreamerPolicy(lidar_env, wc)
    sw, enc = _abi.RdDreamerWeights(), _abi.RdDreamerConvEncoder()
    with pytest.raises(RuntimeError, match="RD_OBS_OCCUPANCY"):
        lidar_env._check(lidar_env.lib.rd_policy_dreamer_init_occupancy(lidar_env._handle, C.byref(sw), C.byref(enc)))
    lidar_env.close()
