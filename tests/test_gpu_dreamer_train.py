"""GPU: the training-mode Dreamer agent step (rd_policy_dreamer_train / rd_rollout_dreamer_train, k_actor_train) and the
in-place weight refresh (rd_policy_dreamer_set_weights, k_pack_weights), through DreamerPolicy.

Bars.  The RSSM and actor head use test_gpu_dreamer's bars (per precision).  The sample a = tanh(mean + sd e1) moves by
at most |d mean| + |e1| |d sd|, so it gets the head bar times (1 + |e1|).  The exploration is checked bit for bit from
the kernel's own a.  The Philox path is compared with the explicit path fed with the float64 Box-Muller restatement of
the same Philox blocks (test_cpu_dreamer_train); the kernel's float32 logf / sqrtf / sincospif put a few ulp on each
normal, so actions of the two paths agree to 1e-3 (the tf32x3 actor-head bar) rather than bitwise."""
import numpy as np
import pytest

from oracle import dreamer_policy as dp
from test_cpu_dreamer_train import posterior_normals, sample, train_normals, train_step
from test_gpu_dreamer import BARS, close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(scope="module")
def austria():
    from racing_dreamer_b200.policy import load_dreamer_checkpoint
    return load_dreamer_checkpoint("austria_dreamer")


def make_env(**kw):
    from racing_dreamer_b200 import BatchedRaceEnv, EnvConfig
    base = dict(tracks=("austria",), action_repeat=4, reset_mode="random", seed=3)
    base.update(kw)
    return BatchedRaceEnv(EnvConfig(**base), device="cuda:0")


def weights_of(kind, austria):
    return austria if kind == "austria" else dp.random_weights(41, normalized=(kind == "random_bn"))


def f32(x):
    return np.asarray(x, np.float32)


def explored(a, amount, e2):
    """what k_actor_train must return, bit for bit: clip(f32(a) + f32(amount) * f32(e2), -1, 1) in float32"""
    return np.clip(f32(a) + np.float32(amount) * f32(e2), np.float32(-1), np.float32(1))


def random_state(rng, n):
    return (rng.standard_normal((n, 30)), rng.uniform(-1, 1, (n, 200)), rng.uniform(-1, 1, (n, 2)))


@pytest.mark.parametrize("precision", ["tf32x3", "tf32"])
@pytest.mark.parametrize("kind", ["austria", "random", "random_bn"])
def test_teacher_forced_training_step(torch_cuda, austria, kind, precision):
    """explicit e: RSSM, actor head and sample against the float64 oracle; exploration bit for bit; state = a'"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 300
    w = weights_of(kind, austria)
    env = make_env(n_envs=n)
    scans = env.reset()["lidar"].clone()
    pol = DreamerPolicy(env, w, noise="explicit", precision=precision)
    rtol, atol, head = BARS[precision]
    rng = np.random.RandomState(5)
    for step in range(2):
        state = random_state(rng, n)
        pol.set_state(*[torch.from_numpy(f32(s)) for s in state])
        es, e1, e2 = f32(rng.standard_normal((n, 30))), f32(rng.standard_normal((n, 2))), f32(rng.standard_normal((n, 2)))
        amount = pol.exploration_amount()
        act = pol.act(scans, torch.from_numpy(es), training=True, eps_sample=torch.from_numpy(e1),
                      eps_expl=torch.from_numpy(e2), debug=True).cpu().numpy()
        d = {k: v.cpu().numpy() for k, v in pol.diagnostics().items()}
        st, de, ac = (t.cpu().numpy() for t in pol.get_state())
        state32 = tuple(s.astype(np.float32).astype(np.float64) for s in state)
        _, new_state, ref = train_step(w, scans.cpu().numpy(), state32, es, e1, e2, float(amount))
        close("mean", d["mean"], ref["mean"], rtol, atol)
        close("deter", de, new_state[1], rtol, atol)
        close("stoch", st, new_state[0], rtol, atol)
        close("actor_mean", d["actor_mean"], ref["actor_mean"], rtol * head, atol * head, dp.MEAN_SCALE)
        close("actor_std", d["actor_std"], ref["actor_std"], rtol * head, atol * head, dp.MEAN_SCALE)
        bar = (atol + rtol * dp.MEAN_SCALE) * head * (1 + np.abs(e1))
        assert (np.abs(d["action"] - ref["sample"]) <= bar).all(), np.abs(d["action"] - ref["sample"]).max()
        # the kernel's sample and log-probability from its own mean / sd (float32 arithmetic)
        m, s = d["actor_mean"].astype(np.float64), d["actor_std"].astype(np.float64)
        a64, lp64 = sample(m, s, e1.astype(np.float64))
        assert np.abs(d["action"] - a64).max() < 2e-5 * (1 + np.abs(e1).max())
        assert np.abs(d["logp"] - lp64).max() < 1e-3 * max(1.0, np.abs(lp64).max()) and (d["index"] == 0).all()
        # exploration bit for bit from the debug record's a, with the schedule's float32 amount
        assert np.array_equal(act, explored(d["action"], amount, e2))
        assert pol.env_steps == (step + 1) * n * 4
        assert np.abs(ac - act).max() <= (2.0 ** -20 if precision == "tf32x3" else 2.0 ** -10)
    env.close()


def test_schedule_and_env_steps_on_the_device(torch_cuda, austria):
    """decay + floor; eval steps leave env_steps; a resumed counter is honoured; multi-car accounting"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    from racing_dreamer_b200.policy import env_steps_per_training_step, exploration_amount
    for n, cars in ((256, 1), (96, 3)):
        env = make_env(n_envs=n, agents_per_world=cars, reset_mode="grid" if cars > 1 else "random", action_repeat=8)
        scans = env.reset()["lidar"].clone()
        per = env_steps_per_training_step(env.cfg)
        pol = DreamerPolicy(env, austria, noise="explicit", expl_amount=0.4, expl_decay=2.5 * per, expl_min=0.1)
        rng = np.random.RandomState(1)
        es, ea = torch.zeros((n, 30)), torch.zeros((n, 100, 2))
        steps = 0
        for k, kind in enumerate(["train", "eval", "train", "train", "eval", "train", "train", "train"]):
            if k == 4:
                pol.env_steps = steps = 17 * per   # resume: the schedule continues from the restored counter
            if kind == "eval":
                pol.act(scans, es, ea)
                assert pol.env_steps == steps
                continue
            e1, e2 = f32(rng.standard_normal((n, 2))), f32(rng.standard_normal((n, 2)))
            amount = exploration_amount(0.4, 2.5 * per, 0.1, steps)
            act = pol.act(scans, es, training=True, eps_sample=torch.from_numpy(e1), eps_expl=torch.from_numpy(e2),
                          debug=True).cpu().numpy()
            assert np.array_equal(act, explored(pol.diagnostics()["action"].cpu().numpy(), amount, e2)), (k, amount)
            steps += n * 8
            assert pol.env_steps == steps
        assert amount == np.float32(0.1)
        env.close()


def test_philox_training_draws(torch_cuda, austria):
    """the Philox path == the explicit path fed with the restated normals; exploration offsets ~ N(0, amount^2)"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n, amount = 4096, 0.02
    env_p, env_e = make_env(n_envs=n, seed=21), make_env(n_envs=n, seed=21)
    scans = env_p.reset()["lidar"].clone()
    env_e.reset()
    pol_p = DreamerPolicy(env_p, austria, noise="philox", expl_amount=amount)
    pol_e = DreamerPolicy(env_e, austria, noise="explicit", expl_amount=amount)
    seed = int(env_p.cfg.seed)
    offsets = []
    for step in range(6):
        pol_e.set_state(*pol_p.get_state())
        a_p = pol_p.act(scans, training=True, debug=True).clone()
        d_p = {k: v.cpu().numpy() for k, v in pol_p.diagnostics().items()}
        e1, e2 = train_normals(seed, n, step)
        es = posterior_normals(seed, n, step)
        pol_e.act(scans, torch.from_numpy(f32(es)), training=True, eps_sample=torch.from_numpy(f32(e1)),
                  eps_expl=torch.from_numpy(f32(e2)), debug=True)
        d_e = {k: v.cpu().numpy() for k, v in pol_e.diagnostics().items()}
        assert np.abs(d_p["mean"] - d_e["mean"]).max() < 2e-3
        assert np.abs(d_p["action"] - d_e["action"]).max() < 1e-3
        assert np.abs(a_p.cpu().numpy() - pol_e.actions.cpu().numpy()).max() < 1e-3
        a = d_p["action"]
        free = np.abs(a) <= 1 - 6 * amount   # a + amount e2 cannot reach the clip (|e2| < 6)
        offsets.append(((a_p.cpu().numpy() - a) / amount)[free])
    o = np.concatenate(offsets)
    assert o.size > 2000, o.size
    # offset / amount ~ N(0, 1): sample mean and std within ~4 standard errors
    assert abs(o.mean()) < 4 / np.sqrt(o.size) and abs(o.std() - 1.0) < 3 / np.sqrt(o.size), (o.size, o.mean(), o.std())
    env_p.close()
    env_e.close()


def test_training_rollout_equals_stepwise(torch_cuda, austria):
    """rd_rollout_dreamer_train == n x (act(training=True) -> env.step) bit for bit; recorded rollout == act + store.step"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    from racing_dreamer_b200.episodes import DeviceEpisodeStore
    n, steps = 1024, 40
    outs = []
    for mode in ("rollout", "stepwise"):
        env = make_env(n_envs=n, seed=6, auto_reset=True)
        env.reset()
        pol = DreamerPolicy(env, austria, noise="philox")
        if mode == "rollout":
            pol.rollout(steps, training=True)
        else:
            for _ in range(steps):
                env.step(pol.act(training=True))
        torch.cuda.synchronize()
        outs.append((env.buf["pose"].clone(), pol.actions.clone()) + tuple(pol.get_state()) + (pol.env_steps,))
        env.close()
    for a, b in zip(outs[0][:-1], outs[1][:-1]):
        assert torch.equal(a, b)
    assert outs[0][-1] == outs[1][-1] == steps * n * 4
    # recorded: the store's rows hold the executed (explored) actions
    from racing_dreamer_b200 import EnvConfig, BatchedRaceEnv
    ec = EnvConfig(tracks=("austria",), n_envs=16, action_repeat=4, auto_reset=False, reset_mode="random",
                   time_limit_steps=30, seed=11)
    runs = []
    for mode in ("rollout", "loop"):
        env = BatchedRaceEnv(ec, device="cuda:0")
        store = DeviceEpisodeStore(env, capacity_rows=400)
        pol = DreamerPolicy(env, austria, noise="philox")
        store.reset()
        executed = set()
        if mode == "rollout":
            pol.rollout(70, training=True, store=store)
        else:
            for _ in range(70):
                a = pol.act(training=True)
                executed.update(map(bytes, a.cpu().numpy()))
                store.step(a)
        torch.cuda.synchronize()
        runs.append((store.episodes(), executed, pol.env_steps))
        env.close()
    (e1, _, s1), (e2, executed, s2) = runs
    assert len(e1) == len(e2) >= 16 and s1 == s2 == 70 * 16 * 4
    for x, y in zip(e1, e2):
        for k in x:
            assert np.array_equal(np.asarray(x[k]).view(np.uint8), np.asarray(y[k]).view(np.uint8)), k
        assert all(bytes(r) in executed for r in f32(y["action"][1:]))


def test_eval_mode_untouched(torch_cuda, austria):
    """after training steps, an evaluation step equals, bit for bit, a fresh policy's from the same state and draws"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 512
    env_a, env_b = make_env(n_envs=n, seed=8), make_env(n_envs=n, seed=8)
    scans = env_a.reset()["lidar"].clone()
    env_b.reset()
    pol_a = DreamerPolicy(env_a, austria, noise="philox")
    for _ in range(3):
        pol_a.act(scans, training=True)
    state = [t.clone() for t in pol_a.get_state()]
    pol_b = DreamerPolicy(env_b, austria, noise="philox")
    for pol in (pol_a, pol_b):   # both through set_state: re-splitting hi + lo can move a tie of the TF32 rounding
        pol.set_state(*state)
    rng = np.random.RandomState(4)
    es, ea = torch.from_numpy(f32(rng.standard_normal((n, 30)))), torch.from_numpy(f32(rng.standard_normal((n, 100, 2))))
    out = []
    for pol in (pol_a, pol_b):
        act = pol.act(scans, es, ea, debug=True, noise="explicit").clone()
        out.append((act, pol.debug.clone()) + tuple(t.clone() for t in pol.get_state()))
    for x, y in zip(*out):
        assert torch.equal(x, y)
    env_a.close()
    env_b.close()


def _acts(torch, pol, scans, rng, n):
    """one explicit evaluation step and one explicit + one zero-noise training step from a fixed state"""
    state = [torch.from_numpy(f32(s)) for s in random_state(rng, n)]
    es, ea = torch.from_numpy(f32(rng.standard_normal((n, 30)))), torch.from_numpy(f32(rng.standard_normal((n, 100, 2))))
    e1, e2 = torch.from_numpy(f32(rng.standard_normal((n, 2)))), torch.from_numpy(f32(rng.standard_normal((n, 2))))
    res = []
    pol.set_state(*state)
    res.append(pol.act(scans, es, ea, noise="explicit", debug=True).clone())
    res.append(pol.debug.clone())
    pol.set_state(*state)
    res.append(pol.act(scans, es, training=True, eps_sample=e1, eps_expl=e2, noise="explicit").clone())
    pol.set_state(*state)
    res.append(pol.act(scans, noise="zero", training=True).clone())
    res += [t.clone() for t in pol.get_state()]
    return res


@pytest.mark.parametrize("precision", ["tf32x3", "tf32"])
@pytest.mark.parametrize("kind", ["random", "random_bn"])
def test_refresh_equals_reinit(torch_cuda, austria, kind, precision):
    """load_weights (numpy and CUDA-tensor sources) == a fresh policy on the new weights, bit for bit; state kept"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 300
    w_old = dp.random_weights(5, normalized=(kind == "random_bn"))
    w_new = dp.random_weights(6, normalized=(kind == "random_bn"))
    envs = [make_env(n_envs=n, seed=2) for _ in range(3)]
    scans = envs[0].reset()["lidar"].clone()
    for e in envs[1:]:
        e.reset()
    fresh = DreamerPolicy(envs[0], w_new, precision=precision)
    want = _acts(torch, fresh, scans, np.random.RandomState(9), n)
    for i, src in enumerate(("numpy", "cuda")):
        pol = DreamerPolicy(envs[1 + i], w_old, precision=precision, noise="philox")
        pol.act(scans, training=True)
        before = [t.clone() for t in pol.get_state()]
        steps = pol.env_steps
        if src == "numpy":
            pol.load_weights(w_new)
        else:
            pol.load_weights({k: torch.from_numpy(v).cuda() for k, v in w_new.items()})
        assert pol.env_steps == steps
        for a, b in zip(before, pol.get_state()):
            assert torch.equal(a, b)
        got = _acts(torch, pol, scans, np.random.RandomState(9), n)
        for j, (x, y) in enumerate(zip(got, want)):
            assert torch.equal(x, y), (src, j)
    for e in envs:
        e.close()


def test_refresh_in_rollouts(torch_cuda, austria):
    """a mid-rollout refresh to the same weights changes nothing (Philox counter and state continue); rollout ->
    load_weights -> rollout enqueued without a sync == the synchronised sequence"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n = 1024
    w_dev = {k: torch.from_numpy(v).cuda() for k, v in austria.items()}
    w2 = dp.random_weights(12)
    w2.update({k: austria[k] for k in ("gru_kernel", "gru_recurrent", "gru_bias", "img1_w", "img1_b", "obs1_w", "obs1_b",
                                       "obs2_w", "obs2_b")})   # a new actor on the shipped world model
    w2_dev = {k: torch.from_numpy(v).cuda() for k, v in w2.items()}
    outs = []
    for mode in ("plain", "same", "nosync", "sync"):
        env = make_env(n_envs=n, seed=6, auto_reset=True)
        env.reset()
        pol = DreamerPolicy(env, austria, noise="philox")
        pol.rollout(15, training=True)
        if mode == "same":
            pol.load_weights(w_dev)
        elif mode == "nosync":
            pol.load_weights(w2_dev)
        elif mode == "sync":
            torch.cuda.synchronize()
            pol.load_weights(w2)
            torch.cuda.synchronize()
        pol.rollout(15, training=True)
        torch.cuda.synchronize()
        outs.append((env.buf["pose"].clone(), pol.actions.clone()) + tuple(t.clone() for t in pol.get_state()))
        env.close()
    plain, same, nosync, sync = outs
    for a, b in zip(plain, same):
        assert torch.equal(a, b)
    for a, b in zip(nosync, sync):
        assert torch.equal(a, b)
    assert not torch.equal(plain[1], sync[1])


def test_refresh_rejects_and_changes_nothing(torch_cuda, austria):
    torch = torch_cuda
    import ctypes as C
    from racing_dreamer_b200 import DreamerPolicy, _abi
    n = 128
    env_a, env_b = make_env(n_envs=n, seed=2), make_env(n_envs=n, seed=2)
    scans = env_a.reset()["lidar"].clone()
    env_b.reset()
    pol, ref = DreamerPolicy(env_a, austria), DreamerPolicy(env_b, austria)
    other = dp.random_weights(3)
    bad = []
    bad.append({k: v for k, v in other.items() if k != "obs2_b"})                        # missing key
    bad.append(dict(other, h1_w=other["h1_w"][:, :200]))                               # wrong shape
    bad.append(dict(other, obs1_b=other["obs1_b"][None]))                               # wrong rank
    bad.append(dp.random_weights(3, actor_layers=3))                                    # another layer count
    bad.append(dp.random_weights(3, normalized=True))                                   # BN present
    bad.append(dict(other, hout_b=torch.zeros(4, device="meta")))                       # another device
    bad.append(dict(other, hout_b=np.zeros(4, np.int32)))                               # not float
    for i, w in enumerate(bad):
        with pytest.raises(ValueError):
            pol.load_weights(w)
    with pytest.raises(TypeError):
        pol.load_weights([other])
    # the library's own checks: another precision, host pointers declared as device ones
    s = pol._weights_struct(other, None, lambda a: a.ctypes.data_as(C.c_void_p))
    s.precision = _abi.RD_PRECISION_TF32
    assert env_a.lib.rd_policy_dreamer_set_weights(env_a._handle, C.byref(s), 0, None) == -1
    s = pol._weights_struct(other, None, lambda a: a.ctypes.data_as(C.c_void_p))
    assert env_a.lib.rd_policy_dreamer_set_weights(env_a._handle, C.byref(s), 1, None) == -1
    s.n_samples = 50
    assert env_a.lib.rd_policy_dreamer_set_weights(env_a._handle, C.byref(s), 0, None) == -1
    torch.cuda.synchronize()
    got, want = _acts(torch, pol, scans, np.random.RandomState(1), n), _acts(torch, ref, scans, np.random.RandomState(1), n)
    for x, y in zip(got, want):
        assert torch.equal(x, y)
    env_a.close()
    env_b.close()
