"""GPU: the model-free actor (Sb3Policy: rd_policy_mlp, k_embed_lidar, k_dense<EPI_DENSE_RELU | TANH>, k_dense<EPI_ACTOR>,
k_mlp_head, k_pack_weights<true>) against the float64 restatement oracle/sb3_policy.py at the shapes the C ABI accepts,
under the bar of test_cpu_sb3_shapes (which holds the case table, the inputs and the bar, and checks that one TF32 pass,
a dropped K tail or a packer that ignores the row pitch fail it).  Per case: the deterministic and explicit-noise
evaluation on synthetic scans; the Philox draws at actor step 1 and env_id_offset 12345 against the explicit path fed
their restatement; weight refresh from host arrays and CUDA tensors == a fresh init, bit for bit.  Then the SAC head's
log_std clamp, clamp bounds set through the C ABI, the C-side rejections, re-init of one env handle with another
architecture, and rollout == the act -> step loop at padded widths."""
import ctypes as C

import numpy as np
import pytest

from oracle import sb3_policy as sp
from test_cpu_sb3_policy import mlp_normals
from test_cpu_sb3_shapes import (ALL_CASES, N_SWEEP, case, case_seed, case_weights, check, reference,
                                 synthetic_scans)

pytestmark = pytest.mark.gpu
GID0 = 12345
PHILOX_TOL = 1e-4   # test_gpu_sb3_policy.test_training_mode's: float32 vs float64 Box-Muller of the same block
RD_ERR_INVALID = -1


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


def make_env(n, n_beams=1080, **kw):
    from racing_dreamer_b200 import BatchedRaceEnv
    from racing_dreamer_b200.compat import baselines_config
    base = dict(seed=3, n_beams=n_beams)
    base.update(kw)
    return BatchedRaceEnv(baselines_config("austria", n, **base), device="cuda:0")


def run(torch, pol, lidar, eps=None):
    """one evaluation step (deterministic, or explicit noise eps): (actions, debug record) clones"""
    e = None if eps is None else torch.from_numpy(eps)
    a = pol.act(lidar, deterministic=eps is None, eps=e, debug=True).clone()
    return a, pol.debug.clone()


def as_np(out):
    """(mean, std, action) of run()'s output"""
    a, d = (t.cpu().numpy() for t in out)
    return d[:, 0:2], d[:, 2:4], a


def same_bits(torch, got, want, what):
    for x, y in zip(got, want):
        assert torch.equal(x, y), what


def run_case(torch, name):
    from racing_dreamer_b200.policy import Sb3Policy
    c = ALL_CASES[name]
    seed = case_seed(name)
    n, E, act = c["n_envs"], c["n_beams"], c["activation"]
    sd, w = case_weights(c, seed)
    obs = synthetic_scans(seed, n, E)
    eps = np.random.default_rng(seed + 1).standard_normal((n, 2)).astype(np.float32)
    ref, bars = reference(w, c, obs)
    ref_s = sp.actor(w, c["algo"], act, obs, eps, deterministic=False)
    env = make_env(n, E, env_id_offset=GID0)
    env.reset()
    lidar = torch.from_numpy(obs).cuda()

    # Philox draws at actor step 1 (one step taken first) and env_id_offset 12345
    pol = Sb3Policy(env, sd, activation=act, noise="philox")
    pol.act(lidar, deterministic=False)
    a_p = pol.act(lidar, deterministic=False).cpu().numpy()

    # a second init on the same handle; evaluation against float64 under the bar
    pol = Sb3Policy(env, sd, activation=act, noise="explicit")
    det, sto = run(torch, pol, lidar), run(torch, pol, lidar, eps)
    worst = {"deterministic": check(f"{name} deterministic", as_np(det), ref, bars),
             "explicit noise": check(f"{name} explicit noise", as_np(sto), ref_s, bars, eps)}
    e1 = mlp_normals(int(env.cfg.seed), n, 1, GID0).astype(np.float32)
    a_e = run(torch, pol, lidar, e1)[0].cpu().numpy()
    assert np.abs(a_p - a_e).max() < PHILOX_TOL, f"{name}: Philox vs explicit {np.abs(a_p - a_e).max():.3e}"

    # refresh from other weights == a fresh init, bit for bit (the packer's pitch at every padded width)
    if c["refresh"]:
        other, _ = case_weights(c, seed + 1)
        for src in ("numpy", "cuda"):
            q = Sb3Policy(env, other, activation=act, noise="explicit")
            assert not torch.equal(run(torch, q, lidar)[1], det[1])
            q.load_weights(sd if src == "numpy" else {k: torch.from_numpy(v).cuda() for k, v in sd.items()})
            same_bits(torch, run(torch, q, lidar), det, f"{name}: refresh ({src}) vs init, deterministic")
            same_bits(torch, run(torch, q, lidar, eps), sto, f"{name}: refresh ({src}) vs init, explicit noise")
    torch.cuda.synchronize()
    env.close()
    print(f"[{name}: {c['algo']} {act} {c['widths']} beams {E} envs {n}] worst |err| / bar:",
          {k: {q: f"{v:.3f}" for q, v in r.items()} for k, r in worst.items()})


@pytest.mark.parametrize("name", [k for k in ALL_CASES if not k.startswith("sweep")])
def test_architecture_vs_oracle(torch_cuda, name):
    run_case(torch_cuda, name)


@pytest.mark.parametrize("seed", range(N_SWEEP))
def test_seeded_architecture_sweep(torch_cuda, seed):
    run_case(torch_cuda, f"sweep{seed}")


def _sac_case(n=300, n_beams=1080):
    return case("sac", [256, 256], n_beams, n)


@pytest.mark.parametrize("log_std_bias", [40.0, -40.0, 2.0])
def test_log_std_clamp(torch_cuda, log_std_bias):
    """log_std_bias +40: std = e^2 everywhere; -40: e^-20 (the bar is relative there); 2: some rows clamp, some not"""
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy
    c = _sac_case()
    sd, w = case_weights(c, 31, log_std_bias=log_std_bias)
    obs = synthetic_scans(31, c["n_envs"], c["n_beams"])
    raw = sp.actor(w, "sac", "relu", obs, log_std_bounds=(-np.inf, np.inf))[1]
    clamped = (raw >= np.exp(sp.LOG_STD_MAX)) | (raw <= np.exp(sp.LOG_STD_MIN))
    assert clamped.all() if abs(log_std_bias) > 30 else 0.1 < clamped.mean() < 0.9
    ref, bars = reference(w, c, obs)
    env = make_env(c["n_envs"])
    pol = Sb3Policy(env, sd, noise="explicit")
    lidar = torch.from_numpy(obs).cuda()
    got = as_np(run(torch, pol, lidar))
    print(log_std_bias, check(f"log_std_bias {log_std_bias}", got, ref, bars))
    env.close()


@pytest.mark.parametrize("bounds", [(-1.0, -1.0), (-0.5, 0.5)])
def test_clamp_bounds_through_the_c_abi(torch_cuda, bounds):
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy
    c = _sac_case(129)
    sd, w = case_weights(c, 32, log_std_bias=0.5)   # log_std in [0.15, 0.65]: some rows clamp at 0.5
    obs = synthetic_scans(32, c["n_envs"], c["n_beams"])
    ref, bars = reference(w, c, obs, log_std_bounds=bounds)
    env = make_env(c["n_envs"])
    pol = Sb3Policy(env, sd, noise="explicit")
    s = pol._struct(pol.weights, lambda a: a.ctypes.data_as(C.c_void_p))
    s.log_std_min, s.log_std_max = bounds
    assert env.lib.rd_policy_mlp_init(env._handle, C.byref(s)) == 0
    got = as_np(run(torch, pol, torch.from_numpy(obs).cuda()))
    print(bounds, check(f"log_std bounds {bounds}", got, ref, bars))
    if bounds[0] == bounds[1]:
        assert np.all(got[1] == got[1][0, 0])
    env.close()


def test_c_rejections_leave_the_policy_working(torch_cuda):
    """every mlp_check refusal through the C ABI (past Sb3Policy's own checks) returns RD_ERR_INVALID with its reason,
    at init and at refresh; the policy on the env then computes what it did before, bit for bit"""
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy
    n, E = 129, 100
    c = case("sac", [33], E, n)
    sd, w = case_weights(c, 33)
    env = make_env(n, E)
    pol = Sb3Policy(env, sd, noise="explicit")
    obs = synthetic_scans(33, n, E)
    lidar = torch.from_numpy(obs).cuda()
    eps = np.random.default_rng(33).standard_normal((n, 2)).astype(np.float32)
    want = run(torch, pol, lidar) + run(torch, pol, lidar, eps)
    host = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    dev_w = {k: torch.from_numpy(v).cuda() for k, v in pol.weights.items()}
    log_std = np.float32([-0.5, 0.25])

    def good(ptr=host, weights=pol.weights):
        return pol._struct(weights, ptr)

    def edit(**fields):
        s = good()
        for k, v in fields.items():
            if k == "width0":
                s.width[0] = v
            elif k in ("w0", "b0"):
                getattr(s, k[0])[0] = v
            else:
                setattr(s, k, v)
        return s

    def diag(**fields):
        s = edit(head=1, log_std_w=None, log_std_b=None, log_std=host(log_std))   # RD_HEAD_DIAG
        for k, v in fields.items():
            setattr(s, k, v)
        return s

    at_init = [("n_layers", edit(n_layers=0)), ("n_layers", edit(n_layers=5)), ("width[0]", edit(width0=0)),
               ("width[0]", edit(width0=1025)), ("in_features", edit(in_features=96)),
               ("bad activation", edit(activation=2)), ("bad head kind", edit(head=2)),
               ("log_std_min > log_std_max", edit(log_std_min=2.5)),
               ("log_std_min > log_std_max", edit(log_std_min=float("nan"))),
               ("log_std_min > log_std_max", edit(log_std_max=float("nan")))]
    at_init += [("null weight pointer", edit(**{k: None})) for k in ("w0", "b0", "mean_w", "mean_b", "log_std_w",
                                                                     "log_std_b")]
    at_init += [("null weight pointer", diag(log_std=None)), ("null weight pointer", diag(mean_b=None))]
    s = good()
    s.mean_w = dev_w["mean_w"].data_ptr()
    at_init.append(("device memory where host memory is expected", s))
    for reason, s in at_init:
        assert env.lib.rd_policy_mlp_init(env._handle, C.byref(s)) == RD_ERR_INVALID, reason
        assert reason.encode() in env.lib.rd_last_error(env._handle), (reason, env.lib.rd_last_error(env._handle))
    stream = env._stream()
    at_refresh = [("on_device: a weight pointer is not memory", good(), 1),
                  ("device memory where host memory", good(lambda t: C.c_void_p(t.data_ptr()), dev_w), 0),
                  ("differ from the ones", edit(width0=32), 0), ("differ from the ones", edit(log_std_min=-19.0), 0),
                  ("differ from the ones", diag(), 0)]
    for reason, s, on_device in at_refresh:
        assert env.lib.rd_policy_mlp_set_weights(env._handle, C.byref(s), on_device, stream) == RD_ERR_INVALID, reason
        assert reason.encode() in env.lib.rd_last_error(env._handle), (reason, env.lib.rd_last_error(env._handle))
    same_bits(torch, run(torch, pol, lidar) + run(torch, pol, lidar, eps), want, "after the rejected calls")
    # 98 beams: load_sb3_checkpoint takes in_features = 98, the C ABI refuses a scan row that is not a multiple of 4
    env98 = make_env(8, 98)
    with pytest.raises(RuntimeError, match="multiple of 4"):
        Sb3Policy(env98, case_weights(case("sac", [33], 98, 8), 34)[0])
    env98.close()
    env.close()


def test_reinit_with_other_architectures(torch_cuda):
    """[1024, 1024] -> [3] -> [1024, 1024] on one env handle, each against the oracle: no buffer sized for the previous
    architecture is reused"""
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy
    n = 300
    obs = synthetic_scans(35, n, 1080)
    lidar = torch.from_numpy(obs).cuda()
    env = make_env(n)
    for i, widths in enumerate(([1024, 1024], [3], [1024, 1024])):
        c = case("sac", widths, 1080, n)
        sd, w = case_weights(c, 35 + i)
        ref, bars = reference(w, c, obs)
        pol = Sb3Policy(env, sd, noise="explicit")
        check(f"init {i} {widths}", as_np(run(torch, pol, lidar)), ref, bars)
    env.close()


def test_rollout_equals_act_step_loop_at_padded_widths(torch_cuda):
    """rd_rollout_mlp == n x (rd_policy_mlp -> rd_step) bit for bit, SAC tanh [33, 129] (36 / 132 padded), 300 envs"""
    torch = torch_cuda
    from racing_dreamer_b200.policy import Sb3Policy
    sd, _ = case_weights(case("sac", [33, 129], 1080, 300, "tanh"), 36)
    outs = []
    for mode in ("rollout", "loop"):
        env = make_env(300, seed=5, auto_reset=True)
        env.reset()
        pol = Sb3Policy(env, sd, activation="tanh")
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
