"""GPU: the model-free baselines' actors on the device (Sb3Policy: rd_policy_mlp, k_dense<EPI_DENSE_RELU | TANH>,
k_mlp_head) against the float64 restatement oracle/sb3_policy.py, their rollouts and weight refresh, and the uniform
random actions (RandomPolicy: k_random_actions) against their NumPy law, bit for bit.

Bars: the evaluation against float64 is held to test_cpu_sb3_shapes' bar (float32-grade, 8x better than one TF32 pass),
the explicit-noise actions to test_gpu_dreamer's tf32x3 bars; the Philox path is compared with the explicit path fed the
float64 Box-Muller restatement of the same blocks (a few float32 ulp per normal)."""
import numpy as np
import pytest

from oracle import sb3_policy as sp
from test_cpu_sb3_policy import make_sd, mlp_normals, random_actions
from test_cpu_sb3_shapes import check, reference
from test_gpu_dreamer import BARS, close

pytestmark = pytest.mark.gpu
RTOL, ATOL, HEAD = BARS["tf32x3"]
RD_ERR_INVALID = -1


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


def make_env(n, **kw):
    from racing_dreamer_b200 import BatchedRaceEnv
    from racing_dreamer_b200.compat import baselines_config
    base = dict(seed=3)
    base.update(kw)
    return BatchedRaceEnv(baselines_config("austria", n, **base), device="cuda:0")


ARCHS = {"sac256": ("sac", dict(widths=(256, 256))), "ppo64": ("ppo", dict(widths=(64, 64))),
         "ppo_shared": ("ppo", dict(widths=(64, 64), shared=(64,))), "sac400": ("sac", dict(widths=(400, 300))),
         "one_layer": ("sac", dict(widths=(100,))), "four_layers": ("ppo", dict(widths=(128, 96, 64, 36)))}


def scans_of(env, torch, steps=3):
    """scans of a running batch: a few random steps after the reset (not only the start grid)"""
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(steps):
        env.step(torch.rand((env.n, 2), device="cuda", generator=g) * 2 - 1)
    return env.buf["lidar"].clone()


@pytest.mark.parametrize("arch", list(ARCHS))
@pytest.mark.parametrize("n", [1, 127, 129, 4096])
def test_evaluation_matches_restatement(torch_cuda, arch, n):
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy, load_sb3_checkpoint
    algo, kw = ARCHS[arch]
    sd = make_sd(algo, 11, **kw)
    env = make_env(n)
    scans = scans_of(env, torch)
    pol = Sb3Policy(env, sd)
    a = pol.act(scans, deterministic=True, debug=True).cpu().numpy()
    d = {k: v.cpu().numpy() for k, v in pol.diagnostics().items()}
    _, w, meta = load_sb3_checkpoint(sd)
    ref, bars = reference(w, dict(algo=algo, activation=meta["activation"]), scans.cpu().numpy())
    check(arch, (d["mean"], d["std"], a), ref, bars)
    env.close()


@pytest.mark.parametrize("arch", ["sac256", "ppo64"])
def test_training_mode(torch_cuda, arch):
    """Philox normals of block (env_id_offset + env, step, 0, RD_STREAM_MLP), at offsets 0 and 12345"""
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy, load_sb3_checkpoint
    algo, kw = ARCHS[arch]
    sd = make_sd(algo, 12, **kw)
    n = 4096
    _, w, meta = load_sb3_checkpoint(sd)
    for gid0 in (0, 12345):
        env_p, env_e = make_env(n, seed=21, env_id_offset=gid0), make_env(n, seed=21, env_id_offset=gid0)
        scans = scans_of(env_p, torch)
        pol_p, pol_e = Sb3Policy(env_p, sd, noise="philox"), Sb3Policy(env_e, sd, noise="explicit")
        seed = int(env_p.cfg.seed)
        for step in range(3):
            e = mlp_normals(seed, n, step, gid0)
            a_e = pol_e.act(scans, deterministic=False, eps=torch.from_numpy(e.astype(np.float32))).cpu().numpy()
            mean, std, act = sp.actor(w, algo, meta["activation"], scans.cpu().numpy(), e.astype(np.float32),
                                      deterministic=False)
            close("explicit action", a_e, act, rtol=HEAD * RTOL, atol=HEAD * ATOL)
            a_p = pol_p.act(scans, deterministic=False).cpu().numpy()
            assert np.abs(a_p - a_e).max() < 1e-4, np.abs(a_p - a_e).max()
        env_p.close()
        env_e.close()
    if algo == "ppo":   # unclipped in the actions buffer; the env's clip = stepping with clip(a, -1, 1)
        big = make_sd("ppo", 12, widths=(64, 64), log_std=(1.5, 1.5))
        env_c = make_env(n, seed=21)
        scans_of(env_c, torch)
        env_p = make_env(n, seed=21)
        scans_of(env_p, torch)
        pol = Sb3Policy(env_p, big)
        a = pol.act(deterministic=False).clone()
        assert a.abs().max().item() > 1.0
        o1 = env_p.step(a)[0]["lidar"].clone()
        o2 = env_c.step(a.clamp(-1, 1))[0]["lidar"]
        assert torch.equal(o1, o2)
        env_c.close()
        env_p.close()


@pytest.mark.parametrize("arch", ["sac256", "ppo64"])
def test_rollout_equals_act_step_loop(torch_cuda, arch):
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy
    algo, kw = ARCHS[arch]
    sd = make_sd(algo, 13, **kw)
    outs = []
    for mode in ("rollout", "loop"):
        env = make_env(256, seed=5, auto_reset=True)
        env.reset()
        pol = Sb3Policy(env, sd)
        if mode == "rollout":
            pol.rollout(40, deterministic=False)
        else:
            for _ in range(40):
                env.step(pol.act(deterministic=False))
        torch.cuda.synchronize()
        outs.append([env.buf[k].clone() for k in ("lidar", "pose", "reward", "done", "progress")] + [pol.actions.clone()])
        env.close()
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("policy", ["ppo", "ppo_deterministic", "random"])
def test_rollout_store_equals_store_step(torch_cuda, policy):
    torch = torch_cuda
    from racing_dreamer_b200.episodes import DeviceEpisodeStore
    from racing_dreamer_b200.policy import RandomPolicy, Sb3Policy
    sd = make_sd("ppo", 14, widths=(64, 64), log_std=(0.8, 0.8))
    runs = []
    for mode in ("rollout", "loop"):
        env = make_env(16, seed=11, auto_reset=False, time_limit_ticks=120)
        store = DeviceEpisodeStore(env, capacity_rows=400)
        det = policy == "ppo_deterministic"   # RD_STORE_POLICY_MLP (else _MLP_TRAIN)
        pol = RandomPolicy(env) if policy == "random" else Sb3Policy(env, sd)
        store.reset()
        if mode == "rollout":
            if policy == "random":
                pol.rollout(70, store=store)
            else:
                pol.rollout(70, deterministic=det, store=store)
        else:
            for _ in range(70):
                store.step(pol.act() if policy == "random" else pol.act(deterministic=det))
        torch.cuda.synchronize()
        runs.append(store.episodes())
        env.close()
    e1, e2 = runs
    assert len(e1) == len(e2) >= 16
    for x, y in zip(e1, e2):
        for k in x:
            assert np.array_equal(np.asarray(x[k]).view(np.uint8), np.asarray(y[k]).view(np.uint8)), k
    acts = np.concatenate([x["action"][1:] for x in e1])
    if policy == "ppo":
        assert np.abs(acts).max() > 1.0   # the recorded actions are the actor's, unclipped
    elif policy == "random":
        assert acts.min() >= -1.0 and acts.max() < 1.0


def test_refresh(torch_cuda):
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy
    sd0, sd1 = make_sd("sac", 15, widths=(256, 256)), make_sd("sac", 16, widths=(256, 256))
    n = 512
    env_a, env_b = make_env(n, seed=4), make_env(n, seed=4)
    scans = scans_of(env_a, torch)
    pol_a = Sb3Policy(env_a, sd0)
    pol_a.act(scans, deterministic=False)
    pol_a.act(scans, deterministic=False)
    # refresh from CUDA tensors (no host synchronisation) == a fresh init with them, Philox counter continued
    pol_a.load_weights({k: torch.from_numpy(v).cuda() for k, v in sd1.items()})
    pol_b = Sb3Policy(env_b, sd1)
    pol_b.act(scans, deterministic=False)
    pol_b.act(scans, deterministic=False)
    for det in (True, False):
        assert torch.equal(pol_a.act(scans, deterministic=det).clone(), pol_b.act(scans, deterministic=det))
    # refresh to the same weights from host arrays changes nothing
    pol_b.act(scans, deterministic=False)
    pol_a.act(scans, deterministic=False)
    pol_a.load_weights(sd1)
    assert torch.equal(pol_a.act(scans, deterministic=False).clone(), pol_b.act(scans, deterministic=False))
    # rejected refreshes change nothing
    for bad in (make_sd("sac", 17, widths=(256, 128)), make_sd("ppo", 17, widths=(256, 256)),
                {k: v for k, v in sd0.items() if not k.startswith("actor.mu")}):
        with pytest.raises(ValueError):
            pol_a.load_weights(bad)
    assert torch.equal(pol_a.act(scans, deterministic=False).clone(), pol_b.act(scans, deterministic=False))
    env_a.close()
    env_b.close()


def test_refresh_mid_rollout(torch_cuda):
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy
    sd = make_sd("ppo", 18, widths=(64, 64))
    outs = []
    for refresh in (False, True):
        env = make_env(128, seed=6, auto_reset=True)
        env.reset()
        pol = Sb3Policy(env, sd)
        pol.rollout(10, deterministic=False)
        if refresh:
            pol.load_weights({k: torch.from_numpy(v).cuda() for k, v in sd.items()})
        pol.rollout(10, deterministic=False)
        torch.cuda.synchronize()
        outs.append((env.buf["pose"].clone(), pol.actions.clone()))
        env.close()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_random_policy(torch_cuda):
    torch = torch_cuda
    from racing_dreamer_b200 import BatchedRaceEnv, EnvConfig
    from racing_dreamer_b200.policy import RandomPolicy
    for env in (make_env(3000, seed=0x123456789), BatchedRaceEnv(EnvConfig(tracks=("austria",), n_envs=300, seed=77,
                                                                           env_id_offset=1000), device="cuda:0")):
        env.reset()
        pol = RandomPolicy(env)
        seed, gid0 = int(env.cfg.seed), int(env.cfg.env_id_offset)
        for step in range(3):
            a = pol.act().cpu().numpy()
            np.testing.assert_array_equal(a, random_actions(seed, env.n, step, gid0))
            assert a.min() >= -1.0 and a.max() < 1.0
        pol.rollout(2)
        np.testing.assert_array_equal(pol.actions.cpu().numpy(), random_actions(seed, env.n, 4, gid0))
        env.close()


def test_env_checks(torch_cuda):
    import ctypes as C
    from racing_dreamer_b200 import BatchedRaceEnv, EnvConfig, _abi
    from racing_dreamer_b200.policy import Sb3Policy, load_sb3_checkpoint
    sd = make_sd("sac", 19, widths=(32,))
    _, w, meta = load_sb3_checkpoint(sd)
    envs = [BatchedRaceEnv(EnvConfig(tracks=("austria",), n_envs=4), device="cuda:0"),   # the dreamer chain
            make_env(4, clip_actions=False), make_env(4, rescale_actions=True), make_env(4, lidar_dtype="float16"),
            make_env(4, obs_type="lidar_occupancy")]
    for env in envs:
        with pytest.raises(ValueError, match="baselines chain"):
            Sb3Policy(env, sd)
        # the same refusal in C
        s = _abi.RdMlpActor()
        s.n_layers, s.in_features, s.width[0], s.activation, s.head = 1, 1080, 32, _abi.RD_ACT_RELU, _abi.RD_HEAD_SQUASHED
        s.log_std_min, s.log_std_max = -20.0, 2.0
        s.w[0], s.b[0] = w["w0"].ctypes.data, w["b0"].ctypes.data
        s.mean_w, s.mean_b, s.log_std_w, s.log_std_b = (w[k].ctypes.data for k in ("mean_w", "mean_b", "log_std_w", "log_std_b"))
        assert env.lib.rd_policy_mlp_init(env._handle, C.byref(s)) == RD_ERR_INVALID
        assert b"baselines chain" in env.lib.rd_last_error(env._handle)
        env.close()
    good = make_env(4)
    Sb3Policy(good, sd)
    good.close()


def test_multi_car_rows(torch_cuda):
    """agents_per_world = 4: every car gets its own row's action"""
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy, load_sb3_checkpoint
    sd = make_sd("ppo", 20, widths=(64, 64))
    env = make_env(64, agents_per_world=4, reset_mode="random_ball")
    scans = scans_of(env, torch)
    pol = Sb3Policy(env, sd)
    a = pol.act(deterministic=True, debug=True).cpu().numpy()
    d = {k: v.cpu().numpy() for k, v in pol.diagnostics().items()}
    _, w, meta = load_sb3_checkpoint(sd)
    ref, bars = reference(w, dict(algo="ppo", activation=meta["activation"]), scans.cpu().numpy())
    check("multi-car rows", (d["mean"], d["std"], a), ref, bars)
    assert len({bytes(r) for r in a}) > 32
    env.close()
