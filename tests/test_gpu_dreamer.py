"""GPU parity of the on-device Dreamer agent (SURVEY §8-f2) through the C ABI (rd_policy_dreamer*, rd_rollout_dreamer)
against the float64 NumPy restatement of RacingDreamer.action (oracle/dreamer_policy.py) on the committed golden
trajectory of the shipped austria checkpoint and on random weights.

Tolerances.  Products run on the tensor cores in TF32 with float32 accumulation.
* precision 'tf32x3' (default): every operand is split into hi + lo TF32 parts and hi*hi + lo*hi + hi*lo is accumulated
  (~2^-21 relative per product), with the K range cut into groups whose partial sums are added in round-to-nearest
  float32 (the tensor core's own accumulation truncates): float32-grade.  Bar: |got - ref| <= 1e-4 + 2e-5 * max_j |ref_j|
  over the env's row of that quantity for the RSSM (deter, posterior mean/std, stoch), five times that for the actor
  head, whose four 400-unit layers amplify their input's rounding.  Measured on the golden trajectory
  (tools/dreamer_errors.py): deter 5e-6, posterior mean 8e-5 of +-41, actor mean 4e-4 of +-5 -- the same figures a
  float32 NumPy evaluation (what the reference's TensorFlow computes in) shows against float64: 4e-6, 7e-5, 2e-4.
* precision 'tf32' (one pass): unit round-off u = 2^-11; a K-term product carries ~u * sqrt(K) * rms|a_k w_k|, i.e. the
  error scales with the magnitude of the layer's outputs (the shipped agent's posterior means reach +-15), and the
  actor's four 400-unit layers amplify a perturbation of their input about tenfold.  Bar: 4e-3 + 2e-3 * row max|ref|
  on the RSSM quantities, twenty times that on the actor head (measured: 4e-3 deter, 2e-2 posterior mean, 0.12 actor
  mean).
SampleDist.mode() is an argmax over 100 draws: the kernel's choice must either be the oracle's draw or one whose
log-probability is within LP_TIE of the maximum (a near tie)."""
import numpy as np
import pytest

from oracle import dreamer_policy as dp
from racing_dreamer_b200 import _abi

pytestmark = pytest.mark.gpu
BARS = {"tf32x3": (2e-5, 1e-4, 5.0), "tf32": (4 * 2.0 ** -11, 4e-3, 20.0)}   # rtol, atol, actor-head factor
RTOL, ATOL, HEAD = BARS["tf32x3"]
LP_TIE = {"tf32x3": 1e-3, "tf32": 5e-2}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(scope="module")
def weights():
    from racing_dreamer_b200.policy import load_dreamer_checkpoint
    return load_dreamer_checkpoint("austria_dreamer")


def make_env(**kw):
    from racing_dreamer_b200 import BatchedRaceEnv, EnvConfig
    return BatchedRaceEnv(EnvConfig(**kw), device="cuda:0")


def close(name, got, ref, rtol=RTOL, atol=ATOL, floor=0.0):
    """|got - ref| <= atol + rtol * scale, scale = the largest |ref| of the env's row (at least `floor`)"""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    scale = np.abs(ref).max(axis=-1, keepdims=True) if ref.ndim > 1 else np.abs(ref)
    scale = np.maximum(scale, floor)
    err = np.abs(got - ref) - rtol * scale
    assert err.max() <= atol, f"{name}: max |err| {np.abs(got - ref).max():.3e} (bar {atol:.1e} + {rtol:.1e} * row max|ref|)"
    return float(np.abs(got - ref).max())


def check_mode(diag, ref, t=None, precision="tf32x3", tie=1.0):
    """the kernel's argmax is the oracle's, or a near tie under the oracle's log-probabilities (within `tie` x LP_TIE:
    a wider actor-head bar widens the margin with it)"""
    idx = diag["index"].cpu().numpy().astype(np.int64)
    lp_all = ref["logp_all"] if t is None else ref["logp_all"][t]
    ridx = ref["index"] if t is None else ref["index"][t]
    rows = np.arange(idx.shape[0])
    gap = lp_all[rows, ridx] - lp_all[rows, idx]
    assert (gap <= tie * LP_TIE[precision]).all(), f"mode(): picked a draw {gap.max():.3e} below the maximum log-probability"
    return float((idx == ridx).mean())


@pytest.mark.parametrize("precision", ["tf32x3", "tf32"])
def test_golden_teacher_forced(torch_cuda, golden_dir, weights, precision):
    """every golden step from the golden's previous state: posterior, deter, actor head, chosen action"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    g = np.load(golden_dir / "dreamer_policy_golden.npz")
    T, n = g["scans"].shape[:2]
    env = make_env(tracks=("austria",), n_envs=n, action_repeat=4)
    env.reset()
    pol = DreamerPolicy(env, weights, noise="explicit", precision=precision)
    rtol, atol, head = BARS[precision]
    worst = {}
    for t in range(T):
        if t == 0:
            pol.reset()
        else:
            pol.set_state(torch.from_numpy(g["stoch"][t - 1]), torch.from_numpy(g["deter"][t - 1]), torch.from_numpy(g["action"][t - 1]))
        act = pol.act(torch.from_numpy(g["scans"][t]).cuda(), torch.from_numpy(g["eps_stoch"][t]), torch.from_numpy(g["eps_actor"][t]),
                      debug=True)
        d = pol.diagnostics()
        st, de, ac = pol.get_state()
        for k, got in (("mean", d["mean"]), ("std", d["std"]), ("stoch", st), ("deter", de), ("actor_mean", d["actor_mean"]),
                       ("actor_std", d["actor_std"])):
            f, fl = (head, dp.MEAN_SCALE) if k.startswith("actor") else (1.0, 0.0)   # the head's outputs live on +-mean_scale
            worst[k] = max(worst.get(k, 0.0), close(f"step {t} {k}", got.cpu().numpy(), g[k][t], rtol * f, atol * f, fl))
        same = check_mode(d, g, t, precision)
        # the action is tanh of the chosen draw; where the same draw was chosen it must agree like the actor mean does
        eq = d["index"].cpu().numpy().astype(np.int64) == g["index"][t]
        u_ref = np.arctanh(np.clip(g["action"][t][eq], -1 + 1e-12, 1 - 1e-12))
        u_got = np.arctanh(np.clip(act.cpu().numpy()[eq].astype(np.float64), -1 + 1e-7, 1 - 1e-7))
        sat = np.abs(u_ref) > 4.0   # tanh saturates in float32 beyond ~4.5: compare the actions themselves there
        close(f"step {t} pre-tanh action", u_got[~sat], u_ref[~sat], max(rtol * head, 1e-4), max(atol * head, 1e-4), dp.MEAN_SCALE)
        assert np.abs(act.cpu().numpy()[eq][sat] - g["action"][t][eq][sat]).max(initial=0.0) < 1e-3
        # the state keeps the action as TF32 hi (+ lo) parts
        assert (ac - act).abs().max() <= (2.0 ** -20 if precision == "tf32x3" else 2.0 ** -11) and same > 0.9
    print(f"[{precision}] max |err| vs float64 oracle:", {k: f"{v:.2e}" for k, v in worst.items()})


def test_golden_free_running(torch_cuda, golden_dir, weights):
    """six agent steps with the recurrent state carried on the device: TF32 noise must not build up"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    g = np.load(golden_dir / "dreamer_policy_golden.npz")
    T, n = g["scans"].shape[:2]
    env = make_env(tracks=("austria",), n_envs=n, action_repeat=4)
    env.reset()
    pol = DreamerPolicy(env, weights, noise="explicit")
    for t in range(T):
        pol.act(torch.from_numpy(g["scans"][t]).cuda(), torch.from_numpy(g["eps_stoch"][t]), torch.from_numpy(g["eps_actor"][t]), debug=True)
        # the previous action feeds img1: keep the comparison meaningful if a near-tie picked another draw
        pol.set_state(action=torch.from_numpy(g["action"][t].astype(np.float32)))
    st, de, _ = pol.get_state()
    close("deter after 6 steps", de.cpu().numpy(), g["deter"][T - 1], rtol=4 * RTOL, atol=4 * ATOL)
    close("posterior mean after 6 steps", pol.diagnostics()["mean"].cpu().numpy(), g["mean"][T - 1], rtol=4 * RTOL, atol=4 * ATOL)


@pytest.mark.parametrize("normalized", [False, True])
def test_random_weights_partial_tile(torch_cuda, normalized):
    """300 envs (2.3 row tiles), both actor heads, random weights, scans from the env itself"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 300
    w = dp.random_weights(11 + normalized, normalized=normalized)
    env = make_env(tracks=("columbia",), n_envs=n, action_repeat=4, reset_mode="random", seed=3)
    scans = env.reset()["lidar"].clone()
    pol = DreamerPolicy(env, w, noise="explicit")
    rng = np.random.RandomState(5)
    state = (rng.standard_normal((n, 30)), rng.uniform(-1, 1, (n, 200)), rng.uniform(-1, 1, (n, 2)))
    pol.set_state(*[torch.from_numpy(s.astype(np.float32)) for s in state])
    es, ea = rng.standard_normal((n, 30)).astype(np.float32), rng.standard_normal((n, 100, 2)).astype(np.float32)
    state32 = tuple(s.astype(np.float32).astype(np.float64) for s in state)
    act_ref, new_state, ref = dp.policy_step(w, scans.cpu().numpy(), state32, es, ea, np.float64)
    act = pol.act(scans, torch.from_numpy(es), torch.from_numpy(ea), debug=True)
    d = pol.diagnostics()
    st, de, _ = pol.get_state()
    close("mean", d["mean"].cpu().numpy(), ref["mean"])
    close("std", d["std"].cpu().numpy(), ref["std"])
    close("deter", de.cpu().numpy(), new_state[1])
    close("stoch", st.cpu().numpy(), new_state[0])
    close("actor_mean", d["actor_mean"].cpu().numpy(), ref["actor_mean"], RTOL * HEAD, ATOL * HEAD, dp.MEAN_SCALE)
    close("actor_std", d["actor_std"].cpu().numpy(), ref["actor_std"], RTOL * HEAD, ATOL * HEAD, dp.MEAN_SCALE)
    check_mode(d, ref)
    eq = d["index"].cpu().numpy().astype(np.int64) == ref["index"]
    assert eq.mean() > 0.9
    assert np.abs(act.cpu().numpy()[eq] - act_ref[eq]).max() < 1e-3   # |d tanh| <= 1: bounded by the pre-tanh error


def test_zero_noise_and_normalised_scans(torch_cuda, weights):
    """noise='zero': stoch = posterior mean, action = tanh(actor mean); an env that emits r/15 - 0.5 gives the same agent"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 256
    env = make_env(tracks=("austria",), n_envs=n, action_repeat=4, reset_mode="random", seed=9)
    scans = env.reset()["lidar"].clone()
    pol = DreamerPolicy(env, weights, noise="zero")
    act = pol.act(debug=True).clone()
    d = pol.diagnostics()
    st, de, ac = pol.get_state()
    # stoch is stored as a hi + lo pair of TF32 numbers (22 bits)
    assert np.abs(st.cpu().numpy() - d["mean"].cpu().numpy()).max() <= 2.0 ** -21 * np.abs(d["mean"].cpu().numpy()).max() + 1e-7
    assert np.abs(act.cpu().numpy() - np.tanh(d["actor_mean"].cpu().numpy())).max() < 1e-6
    _, new_state, ref = dp.policy_step(weights, scans.cpu().numpy(), None, np.zeros((n, 30)), None, np.float64)
    close("zero-noise deter", de.cpu().numpy(), new_state[1])
    close("zero-noise actor mean", d["actor_mean"].cpu().numpy(), ref["actor_mean"], RTOL * HEAD, ATOL * HEAD, dp.MEAN_SCALE)
    env2 = make_env(tracks=("austria",), n_envs=n, action_repeat=4, reset_mode="random", seed=9, normalize_lidar=True)
    scans2 = env2.reset()["lidar"]
    assert np.abs(scans2.cpu().numpy() - (scans.cpu().numpy() / 15.0 - 0.5)).max() < 1e-6
    pol2 = DreamerPolicy(env2, weights, noise="zero")
    pol2.act(debug=True)
    close("normalised-scan env: actor mean", pol2.diagnostics()["actor_mean"].cpu().numpy(), ref["actor_mean"], RTOL * HEAD, ATOL * HEAD, dp.MEAN_SCALE)
    close("normalised-scan env: posterior mean", pol2.diagnostics()["mean"].cpu().numpy(), ref["mean"])


def test_philox_draws(torch_cuda, weights):
    """the posterior draws are standard normal, differ between envs and steps, and repeat for the same (seed, env, step)"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 4096
    runs = []
    for _ in range(2):
        env = make_env(tracks=("austria",), n_envs=n, action_repeat=4, reset_mode="random", seed=21)
        env.reset()
        pol = DreamerPolicy(env, weights, noise="philox")
        eps, acts = [], []
        for _ in range(2):
            acts.append(pol.act(debug=True).clone())
            d = pol.diagnostics()
            st, _, _ = pol.get_state()
            eps.append(((st - d["mean"]) / d["std"]).cpu().numpy())
        runs.append((eps, acts))
    (e0, a0), (e1, a1) = runs
    assert all(torch.equal(x, y) for x, y in zip(a0, a1)) and all(np.array_equal(x, y) for x, y in zip(e0, e1))
    e = np.concatenate(e0)
    assert abs(e.mean()) < 0.02 and abs(e.std() - 1.0) < 0.03 and abs((e ** 3).mean()) < 0.05
    assert np.abs(e0[0] - e0[1]).mean() > 0.5 and np.abs(e0[0][0] - e0[0][1]).mean() > 0.3
    env = make_env(tracks=("austria",), n_envs=n, action_repeat=4, reset_mode="random", seed=22)
    env.reset()
    pol = DreamerPolicy(env, weights, noise="philox")
    pol.act(debug=True)
    st, _, _ = pol.get_state()
    d = pol.diagnostics()
    assert np.abs(((st - d["mean"]) / d["std"]).cpu().numpy() - e0[0]).mean() > 0.5   # another seed, other draws


def test_state_cleared_on_reset(torch_cuda, weights):
    """`state is None` after an env reset [REF racing_dreamer.py:66-68]: auto-reset inside rd_step and rd_reset(mask)"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 512
    env = make_env(tracks=("treitlstrasse_v2",), n_envs=n, action_repeat=8, reset_mode="random", seed=4, auto_reset=True)
    env.reset()
    pol = DreamerPolicy(env, weights, noise="philox")
    gen = torch.Generator(device="cuda").manual_seed(0)
    seen = 0
    for _ in range(40):
        pol.act()
        rand = torch.rand((n, 2), device="cuda", generator=gen) * 2 - 1   # random driving: collisions within a few steps
        _, _, done, _ = env.step(rand)
        st, de, ac = pol.get_state()
        zero = (st.abs().sum(1) == 0) & (de.abs().sum(1) == 0) & (ac.abs().sum(1) == 0)
        assert torch.equal(zero, done), "exactly the envs that were reset have a cleared agent state"
        seen += int(done.sum())
    assert seen > 20
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[::3] = 1
    pol.act()
    before = [t.clone() for t in pol.get_state()]
    env.reset(mask=mask)
    after = pol.get_state()
    for b, a in zip(before, after):
        assert (a[mask.bool()] == 0).all() and torch.equal(a[~mask.bool()], b[~mask.bool()])


def test_rollout_equals_stepwise(torch_cuda, weights):
    """rd_rollout_dreamer == n x (rd_policy_dreamer -> rd_step), bit for bit, and the shipped agent makes progress"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n, steps = 1024, 60
    outs = []
    for mode in ("rollout", "stepwise"):
        env = make_env(tracks=("austria",), n_envs=n, action_repeat=4, reset_mode="random", seed=6, auto_reset=True)
        env.reset()
        pol = DreamerPolicy(env, weights, noise="philox")
        if mode == "rollout":
            pol.rollout(steps)
        else:
            for _ in range(steps):
                env.step(pol.act())
        torch.cuda.synchronize()
        outs.append((env.buf["pose"].clone(), env.buf["lidar"].clone(), pol.actions.clone(), env.read_stats()))
    for a, b in zip(outs[0][:3], outs[1][:3]):
        assert torch.equal(a, b)
    stats = outs[0][3]
    assert stats["env_steps"] == n * steps and np.isfinite(outs[0][0].cpu().numpy()).all()
    # the reference's trained agent drives in this simulator: far fewer crashes than steps/20 per env (random driving)
    assert stats["episodes"] < 0.5 * n, stats


@pytest.mark.parametrize("n", [300, 5000])
def test_actor_chain_is_bitwise_the_per_layer_launches(torch_cuda, weights, monkeypatch, n):
    """k_dense_chain (the actor trunk in one launch, row-block counters between the layers) == one k_dense launch per
    layer, bit for bit: partial row tile (300 envs) and more row blocks than resident CTA groups (5000 envs = 40)"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    outs = []
    for chain in ("1", "0"):
        monkeypatch.setenv("RD_DREAMER_CHAIN", chain)
        env = make_env(tracks=("austria",), n_envs=n, action_repeat=4, reset_mode="random", seed=9, auto_reset=True)
        env.reset()
        pol = DreamerPolicy(env, weights, noise="philox")
        pol.rollout(12)
        torch.cuda.synchronize()
        outs.append((pol.actions.clone(),) + tuple(t.clone() for t in pol.get_state()) + (env.buf["pose"].clone(),))
        env.close()
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("layers", [1, 2, 3, 5, 6, 7])
def test_actor_trunk_depths_other_than_the_shipped_four(torch_cuda, layers):
    """The C ABI takes 1..7 trunk layers; k_dense_chain runs them four per launch (1 = a launch without any counter,
    2 / 3 = one launch of that many, 5 / 6 / 7 = a launch of four and one of one / two / three).  Random weights,
    explicit noise, against the float64 restatement."""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 700
    w = dp.random_weights(30 + layers, actor_layers=layers)
    env = make_env(tracks=("austria",), n_envs=n, action_repeat=4, reset_mode="random", seed=4)
    scans = env.reset()["lidar"].clone()
    pol = DreamerPolicy(env, w, noise="explicit")
    rng = np.random.RandomState(6)
    state = (rng.standard_normal((n, 30)), rng.uniform(-1, 1, (n, 200)), rng.uniform(-1, 1, (n, 2)))
    pol.set_state(*[torch.from_numpy(s.astype(np.float32)) for s in state])
    es, ea = rng.standard_normal((n, 30)).astype(np.float32), rng.standard_normal((n, 100, 2)).astype(np.float32)
    state32 = tuple(s.astype(np.float32).astype(np.float64) for s in state)
    act_ref, new_state, ref = dp.policy_step(w, scans.cpu().numpy(), state32, es, ea, np.float64)
    for rep in range(2):   # twice: the counters of the second launch start where the first one left them
        pol.set_state(*[torch.from_numpy(s.astype(np.float32)) for s in state])
        pol.act(scans, torch.from_numpy(es), torch.from_numpy(ea), debug=True)
        d = pol.diagnostics()
        close(f"actor_mean (pass {rep})", d["actor_mean"].cpu().numpy(), ref["actor_mean"], RTOL * HEAD, ATOL * HEAD, dp.MEAN_SCALE)
        close(f"actor_std (pass {rep})", d["actor_std"].cpu().numpy(), ref["actor_std"], RTOL * HEAD, ATOL * HEAD, dp.MEAN_SCALE)
    env.close()


def test_error_paths(torch_cuda, weights):
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    env = make_env(tracks=("austria",), n_envs=8, action_repeat=4)
    act = torch.zeros((8, 2), device="cuda")
    rc = env.lib.rd_policy_dreamer(env._handle, env.buf["lidar"].data_ptr(), act.data_ptr(), 0, None, None, None, None)
    assert rc == _abi.ERR_STATE if hasattr(_abi, "ERR_STATE") else rc == -3
    env2 = make_env(tracks=("austria",), n_envs=8, action_repeat=4, n_beams=540)
    with pytest.raises(ValueError):
        DreamerPolicy(env2, weights)
    with pytest.raises(NotImplementedError):
        DreamerPolicy(env, weights, actor_version="bogus")
    with pytest.raises(ValueError):
        DreamerPolicy(env, weights, actor_version="normalized")
    pol = DreamerPolicy(env, weights, noise="explicit")
    env.reset()
    with pytest.raises(ValueError):
        pol.act()
    with pytest.raises(RuntimeError):
        env._check(env.lib.rd_rollout_dreamer(env._handle, 1, None, None, 1, None))
