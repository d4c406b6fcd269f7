"""GPU: the Dreamer agent kernels (rd_gemm.cuh k_dense, k_dense_chain, k_actor_mode, k_actor_train, k_pack_weights, driven
by rd_dreamer.cuh) against the float64 restatement (oracle/dreamer_policy.py) at architectures, sample counts and batch
sizes other than the shipped one (deter 200, hidden 200, units 400, embed 1080, 100 samples).  The C ABI takes stoch 30;
deter, hidden, actor units and embed = n_beams positive multiples of 4; 1..7 trunk layers; n_samples >= 1; any number
of envs.  What the chosen values reach (64-wide k_dense tiles, 128-wide k_dense_chain tiles, 32-wide K blocks):
  * width 4: every layer's K is one partial block; units <= 32: a chain layer is one K block; units <= 128: the chain
    runs as clusters of one CTA; deter < 64: the GRU's three gate slabs (W rows 0, D, 2D) fall in one N tile;
  * 128 / 256 / 512 / 2048: exact tile multiples, no tail anywhere;
  * hidden 1028: 17 N tiles of img1 / obs1 (the last one 4 columns wide) and a 40-block GRU K chain;
  * units 1028: 9 N tiles, more than a cluster may hold: k_dense_chain runs without clusters (tf32x3 mode only chains);
  * 2, 3, 5, 7 layers: chain launches of 2, 3, 4 + 1 and 4 + 3 layers;
  * n_samples 1, 3, 255, 256, 257, 1000: k_actor_mode's odd tails and the draws beyond the 4 x 64 it makes before
    griddepcontrol.wait;  1, 127, 128, 129, 300 envs: around the 128-row tiles.

Bars.  test_gpu_dreamer's, per precision, widened only where a shape's K chains are longer than the shipped ones, by
that module's error model:
  * tf32x3: the truncating accumulation drifts in proportion to the K blocks one accumulator group takes in.  Per layer
    f = ceil(blocks / groups) / (the same for the shipped layer), groups cut as dr_build cuts them.  Shipped: img1 1,
    GRU 14 (7 + 7 blocks, one group), obs1 6 (41 blocks in 7 groups), obs2 4, h0 4, h1.. and hout 5.
  * tf32: u sqrt(K) per layer, f = sqrt(K / shipped K).
  A quantity's bars (rtol and atol) are multiplied by the largest f (at least 1) of the layers in front of it: deter
  <- img1, GRU; posterior mean / std / stoch <- + obs1, obs2; actor head <- + trunk, hout.  The near-tie margin of
  mode() takes the head's factor (a log-probability moves with the head's mean and sd).  An action whose draw e is the
  oracle's moves by at most |d mean| + |e| |d sd|: the head bar times (1 + |e|).  The free-running second step, whose
  state carries the first step's error, gets 4x the bars (test_golden_free_running's margin for carried state).
Second, model-free yardstick (tf32x3, teacher-forced step): the oracle evaluated in float32, what the reference's
TensorFlow computes in.  An x3 product carries ~2^-21 relative error and a float32 one 2^-24, so the kernel's largest
error against float64 must stay within 8x the float32 evaluation's, plus the documented absolute floor (1e-4; 5e-4 on
the actor head)."""
import math

import numpy as np
import pytest

from oracle import dreamer_policy as dp
from test_cpu_dreamer_train import actor_normals, posterior_normals, train_step
from test_gpu_dreamer import BARS, check_mode, close
from test_gpu_dreamer_train import explored

pytestmark = pytest.mark.gpu
SHIPPED = dict(deter=200, hidden=200, units=400, embed=1080)
F32_MULTIPLE = 8.0   # 2^-21 / 2^-24
FREE_RUNNING = 4.0
QUANTITY_STAGE = {"deter": 0, "mean": 1, "std": 1, "stoch": 1, "actor_mean": 2, "actor_std": 2}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    torch.cuda.set_device(0)
    return torch


def make_env(n_envs, n_beams, **kw):
    from racing_dreamer_b200 import BatchedRaceEnv, EnvConfig
    base = dict(tracks=("austria",), action_repeat=4, reset_mode="random", seed=3)
    base.update(kw)
    return BatchedRaceEnv(EnvConfig(n_envs=n_envs, n_beams=n_beams, **base), device="cuda:0")


def f32(x):
    return np.asarray(x, np.float32)


def _blocks(k):
    return -(-k // 32)


def _per_group(blocks, max_groups):
    """the longest accumulator group of a dense layer's hi*hi K chain (dr_build: ~6 blocks per group, at most max_groups)"""
    groups = max(1, min(max_groups, (blocks + 5) // 6))
    return -(-blocks // groups)


def _layer_chains(deter, hidden, units, embed, precision):
    """per stage (deter, posterior, actor head): the layers' K-chain measure -- x3: blocks per accumulator group,
    tf32: K"""
    D, H, U, E = deter, hidden, units, embed
    if precision == "tf32x3":
        return [[1, _blocks(H) + _blocks(D)],                                        # img1, GRU (one main group)
                [_per_group(_blocks(D) + _blocks(E), 7), _per_group(_blocks(H), 3)],   # obs1, obs2
                [_per_group(_blocks(32 + D), 3), _per_group(_blocks(U), 3)]]          # h0, h1.. / hout
    return [[32, H + D], [D + E, H], [32 + D, U]]


def bar_factors(deter, hidden, units, embed, precision):
    """[deter, posterior, actor head] factors of the module docstring's error model"""
    got, ship = _layer_chains(deter, hidden, units, embed, precision), _layer_chains(**SHIPPED, precision=precision)
    out, f = [], 1.0
    for g, s in zip(got, ship):
        for a, b in zip(g, s):
            f = max(f, a / b if precision == "tf32x3" else math.sqrt(a / b))
        out.append(f)
    return out


def random_state(rng, n, deter):
    return f32(rng.standard_normal((n, 30))), f32(rng.uniform(-1, 1, (n, deter))), f32(rng.uniform(-1, 1, (n, 2)))


def scans_of(rng, n, embed, normalised):
    """raw scans past both ends of the [0, 15] clip, and what the kernel reads (r/15 - 0.5 if the env normalises)"""
    import torch
    scan = f32(rng.uniform(-1.0, 20.0, (n, embed)))
    return scan, torch.from_numpy(dp.preprocess_lidar(scan) if normalised else scan).cuda()


def explicit_step(torch, pol, lidar, state, es, ea):
    """one explicit-noise evaluation step from `state`: (action, debug record, stoch, deter, previous action) clones"""
    pol.set_state(*[torch.from_numpy(s) for s in state])
    act = pol.act(lidar, torch.from_numpy(es), torch.from_numpy(ea), debug=True).clone()
    return [act, pol.debug.clone()] + [t.clone() for t in pol.get_state()]


def train_once(torch, pol, lidar, state, es, e1, e2):
    pol.set_state(*[torch.from_numpy(s) for s in state])
    act = pol.act(lidar, torch.from_numpy(es), training=True, eps_sample=torch.from_numpy(e1), eps_expl=torch.from_numpy(e2),
                  debug=True).clone()
    return [act, pol.debug.clone()] + [t.clone() for t in pol.get_state()]


def same_bits(torch, got, want, what):
    for j, (x, y) in enumerate(zip(got, want)):
        assert torch.equal(x, y), f"{what}: output {j} differs"


def compare_step(act, d, st, de, act_ref, ref, new_state, ea, precision, fac, ref32=None, state32=None):
    """one evaluation step against the float64 oracle (bars x fac per stage); with ref32: the float32 yardstick too.
    Returns {quantity: max |err|} (and '<quantity>/f32' for the float32 evaluation's)."""
    rtol, atol, head = BARS[precision]
    got = dict(mean=d["mean"], std=d["std"], stoch=st, deter=de, actor_mean=d["actor_mean"], actor_std=d["actor_std"])
    want = dict(mean=ref["mean"], std=ref["std"], stoch=new_state[0], deter=new_state[1], actor_mean=ref["actor_mean"],
                actor_std=ref["actor_std"])
    worst = {}
    for k in got:
        f = fac[QUANTITY_STAGE[k]]
        h, fl = (head, dp.MEAN_SCALE) if k.startswith("actor") else (1.0, 0.0)
        worst[k] = close(k, got[k], want[k], rtol * h * f, atol * h * f, fl)
        if ref32 is not None:
            w32 = dict(mean=ref32["mean"], std=ref32["std"], stoch=state32[0], deter=state32[1],
                       actor_mean=ref32["actor_mean"], actor_std=ref32["actor_std"])[k]
            e32 = float(np.abs(np.asarray(w32, np.float64) - want[k]).max())
            worst[k + "/f32"] = e32
            assert worst[k] <= F32_MULTIPLE * e32 + atol * h, f"{k}: {worst[k]:.3e} vs float32 evaluation {e32:.3e}"
    # where the kernel chose the oracle's draw, the action is tanh of it: |d a| <= |d mean| + |e| |d sd|
    n = act.shape[0]
    idx = d["index"].astype(np.int64)
    eq = idx == ref["index"]
    e_sel = np.abs(ea[np.arange(n), ref["index"]]).max(-1)
    scale = np.maximum(dp.MEAN_SCALE, np.maximum(np.abs(want["actor_mean"]).max(-1), np.abs(want["actor_std"]).max(-1)))
    bar = (atol + rtol * scale) * head * fac[2] * (1.0 + e_sel)
    err = np.abs(act.astype(np.float64) - act_ref).max(-1)
    assert (err[eq] <= bar[eq]).all(), f"action: {err[eq].max():.3e} where the oracle's draw was chosen"
    worst["action"] = float(err[eq].max(initial=0.0))
    worst["same draw"] = float(eq.mean())
    return worst


def run_case(torch, monkeypatch, deter, hidden, units, layers, embed, n_samples, n_envs, precision="tf32x3",
             normalized=False, norm_scan=False, refresh=False, seed=0):
    from racing_dreamer_b200 import DreamerPolicy
    D, S, n = deter, n_samples, n_envs
    x3 = precision == "tf32x3"
    fac = bar_factors(deter, hidden, units, embed, precision)
    w = dp.random_weights(100 + seed, n_beams=embed, normalized=normalized, actor_layers=layers, deter=deter,
                          hidden=hidden, units=units)
    env = make_env(n, embed, normalize_lidar=norm_scan)
    rng = np.random.RandomState(seed)
    scan, lidar = scans_of(rng, n, embed, norm_scan)
    pol = DreamerPolicy(env, w, noise="explicit", n_samples=S, precision=precision)
    tag = f"[{precision} D{deter} H{hidden} U{units} L{layers} E{embed} S{S} N{n}{' bn' if normalized else ''}]"

    # 1. teacher-forced step from a random latent state
    state = random_state(rng, n, D)
    es, ea = f32(rng.standard_normal((n, 30))), f32(rng.standard_normal((n, S, 2)))
    first = explicit_step(torch, pol, lidar, state, es, ea)
    diag = pol.diagnostics()
    d = {k: v.cpu().numpy() for k, v in diag.items()}
    act, st, de, ac = (t.cpu().numpy() for t in (first[0], first[2], first[3], first[4]))
    s64 = tuple(s.astype(np.float64) for s in state)
    act_ref, new_state, ref = dp.policy_step(w, scan, s64, es, ea, np.float64)
    _, state32, ref32 = dp.policy_step(w, scan, state, es, ea, np.float32)
    worst = compare_step(act, d, st, de, act_ref, ref, new_state, ea, precision, fac, *((ref32, state32) if x3 else ()))
    check_mode(diag, ref, precision=precision, tie=fac[2])
    assert np.abs(ac - act).max() <= (2.0 ** -20 if x3 else 2.0 ** -11)   # the state keeps the action as TF32 hi (+ lo)

    # 2. a free-running second step: the latent stays on the device (ping-pong rows); the previous action is the
    #    oracle's, so that a near tie in step 1 does not change what img1 reads
    pol.set_state(action=torch.from_numpy(f32(act_ref)))
    es2, ea2 = f32(rng.standard_normal((n, 30))), f32(rng.standard_normal((n, S, 2)))
    act2 = pol.act(lidar, torch.from_numpy(es2), torch.from_numpy(ea2), debug=True).cpu().numpy()
    diag2 = pol.diagnostics()
    d2 = {k: v.cpu().numpy() for k, v in diag2.items()}
    st2, de2, _ = (t.cpu().numpy() for t in pol.get_state())
    act_ref2, new_state2, ref2 = dp.policy_step(w, scan, (new_state[0], new_state[1], f32(act_ref).astype(np.float64)), es2,
                                                ea2, np.float64)
    worst2 = compare_step(act2, d2, st2, de2, act_ref2, ref2, new_state2, ea2, precision, [FREE_RUNNING * f for f in fac])
    check_mode(diag2, ref2, precision=precision, tie=FREE_RUNNING * fac[2])

    # 3. tf32x3: k_dense_chain == one k_dense launch per trunk layer, bit for bit
    if x3:
        with monkeypatch.context() as m:
            m.setenv("RD_DREAMER_CHAIN", "0")
            per_layer = DreamerPolicy(env, w, noise="explicit", n_samples=S, precision=precision)
        same_bits(torch, explicit_step(torch, per_layer, lidar, state, es, ea), first, f"{tag} chain vs per-layer launches")

    # 4. weight refresh (host and CUDA sources) == a fresh policy; one training-mode step, exploration bit for bit
    if refresh:
        e1, e2 = f32(rng.standard_normal((n, 2))), f32(rng.standard_normal((n, 2)))
        fresh = DreamerPolicy(env, w, noise="explicit", n_samples=S, precision=precision)
        amount = fresh.exploration_amount()
        trained = train_once(torch, fresh, lidar, state, es, e1, e2)
        dt = {k: v.cpu().numpy() for k, v in fresh.diagnostics().items()}
        _, tstate, tref = train_step(w, scan, s64, es, e1, e2, float(amount))
        rtol, atol, head = BARS[precision]
        close("train: mean", dt["mean"], tref["mean"], rtol * fac[1], atol * fac[1])
        close("train: deter", trained[3].cpu().numpy(), tstate[1], rtol * fac[0], atol * fac[0])
        close("train: actor_mean", dt["actor_mean"], tref["actor_mean"], rtol * head * fac[2], atol * head * fac[2], dp.MEAN_SCALE)
        close("train: actor_std", dt["actor_std"], tref["actor_std"], rtol * head * fac[2], atol * head * fac[2], dp.MEAN_SCALE)
        bar = (atol + rtol * dp.MEAN_SCALE) * head * fac[2] * (1 + np.abs(e1))
        assert (np.abs(dt["action"] - tref["sample"]) <= bar).all(), np.abs(dt["action"] - tref["sample"]).max()
        assert np.array_equal(trained[0].cpu().numpy(), explored(dt["action"], amount, e2))
        other = dp.random_weights(200 + seed, n_beams=embed, normalized=normalized, actor_layers=layers, deter=deter,
                                  hidden=hidden, units=units)
        for src in ("numpy", "cuda"):
            q = DreamerPolicy(env, other, noise="explicit", n_samples=S, precision=precision)
            q.load_weights(w if src == "numpy" else {k: torch.from_numpy(v).cuda() for k, v in w.items()})
            same_bits(torch, explicit_step(torch, q, lidar, state, es, ea), first, f"{tag} refresh ({src}) vs init")
            same_bits(torch, train_once(torch, q, lidar, state, es, e1, e2), trained, f"{tag} refresh ({src}), training step")
    torch.cuda.synchronize()
    env.close()
    print(tag, "max |err| vs float64 (and of the float32 evaluation):", {k: f"{v:.2e}" for k, v in worst.items()},
          "second step:", {k: f"{v:.2e}" for k, v in worst2.items()})


# hand-picked: each names the path it reaches (module docstring)
CASES = {
    "width4_x3":            dict(deter=4, hidden=4, units=4, layers=2, embed=4, n_samples=3, n_envs=129),
    "width4_tf32_bn":       dict(deter=4, hidden=28, units=4, layers=3, embed=100, n_samples=1, n_envs=127,
                                 precision="tf32", normalized=True),
    "one_env":              dict(deter=36, hidden=100, units=132, layers=5, embed=360, n_samples=257, n_envs=1),
    "exact_tiles":          dict(deter=128, hidden=256, units=512, layers=3, embed=2048, n_samples=256, n_envs=128,
                                 refresh=True),
    "chain_without_clusters": dict(deter=100, hidden=300, units=1028, layers=3, embed=360, n_samples=64, n_envs=300),
    "hidden1028_layers7":   dict(deter=212, hidden=1028, units=516, layers=7, embed=2048, n_samples=1000, n_envs=128,
                                 refresh=True, normalized=True),
    "deter36_single_block_chain": dict(deter=36, hidden=28, units=32, layers=2, embed=100, n_samples=255, n_envs=300,
                                       normalized=True, norm_scan=True),
    "deter516_units516_layers5": dict(deter=516, hidden=100, units=516, layers=5, embed=4, n_samples=256, n_envs=129),
    "tf32_units1028":       dict(deter=212, hidden=300, units=1028, layers=2, embed=360, n_samples=64, n_envs=300,
                                 precision="tf32", norm_scan=True, refresh=True),
    "tf32_hidden1028":      dict(deter=516, hidden=1028, units=132, layers=7, embed=2048, n_samples=1000, n_envs=129,
                                 precision="tf32"),
    "units400_layers3_bn":  dict(deter=100, hidden=4, units=400, layers=3, embed=100, n_samples=3, n_envs=127,
                                 normalized=True, refresh=True),
}


@pytest.mark.parametrize("name", list(CASES))
def test_architecture_vs_oracle(torch_cuda, monkeypatch, name):
    run_case(torch_cuda, monkeypatch, seed=len(name), **CASES[name])


def _sweep_case(seed):
    r = np.random.RandomState(5000 + seed)
    c = dict(deter=int(r.choice([4, 36, 100, 212, 516])), hidden=int(r.choice([4, 28, 100, 300, 1028])),
             units=int(r.choice([4, 32, 132, 400, 516, 1028])), layers=int(r.choice([2, 3, 5, 7])),
             embed=int(r.choice([4, 100, 360, 2048])), n_samples=int(r.choice([1, 3, 64, 255, 256, 257, 1000])),
             n_envs=int(r.choice([1, 127, 128, 129, 300])), precision=str(r.choice(["tf32x3", "tf32x3", "tf32"])),
             normalized=bool(r.rand() < 0.4), norm_scan=bool(r.rand() < 0.25), refresh=bool(r.rand() < 0.25))
    return c


@pytest.mark.parametrize("seed", range(16))
def test_seeded_architecture_sweep(torch_cuda, monkeypatch, seed):
    run_case(torch_cuda, monkeypatch, seed=seed, **_sweep_case(seed))


@pytest.mark.parametrize("n_samples", [3, 100, 256, 257, 1000])
def test_philox_evaluation_draws(torch_cuda, n_samples):
    """k_actor_mode's Philox draws (block (gid0 + env, step, s - s % 2, RD_STREAM_ACTOR), normals 2 (s % 2) + d) and the
    posterior's, at step 1 and env_id_offset 12345: the Philox policy == an explicit-noise policy fed the restated
    draws from the same state (the same draw, or a near tie under the oracle's log-probabilities; actions within the
    tf32x3 head bar, 1e-3, where the same draw was chosen)"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n, gid0, S = 300, 12345, n_samples
    deter, hidden, units, embed, layers = 36, 100, 132, 100, 3
    w = dp.random_weights(9, n_beams=embed, actor_layers=layers, deter=deter, hidden=hidden, units=units)
    env = make_env(n, embed, env_id_offset=gid0, seed=77)
    seed = int(env.cfg.seed)
    rng = np.random.RandomState(S)
    scan, lidar = scans_of(rng, n, embed, False)
    state = random_state(rng, n, deter)
    pol = DreamerPolicy(env, w, noise="philox", n_samples=S)
    pol.act(lidar)   # step 0
    pol.set_state(*[torch.from_numpy(s) for s in state])
    act_p = pol.act(lidar, debug=True).cpu().numpy()
    d_p = pol.diagnostics()
    idx_p = d_p["index"].cpu().numpy().astype(np.int64)
    mean_p = d_p["mean"].cpu().numpy()
    es, ea = f32(posterior_normals(seed, n, 1, gid0)), f32(actor_normals(seed, n, 1, S, gid0))
    _, _, ref = dp.policy_step(w, scan, tuple(s.astype(np.float64) for s in state), es, ea, np.float64)
    check_mode(d_p, ref)
    exp = DreamerPolicy(env, w, noise="explicit", n_samples=S)
    out = explicit_step(torch, exp, lidar, state, es, ea)
    d_e = exp.diagnostics()
    check_mode(d_e, ref)
    assert np.abs(mean_p - d_e["mean"].cpu().numpy()).max() < 2e-3
    eq = idx_p == d_e["index"].cpu().numpy().astype(np.int64)
    assert eq.mean() > 0.9, eq.mean()
    assert np.abs(act_p[eq] - out[0].cpu().numpy()[eq]).max() < 1e-3
    env.close()


def test_rollout_equals_stepwise_at_another_architecture(torch_cuda):
    """rd_rollout_dreamer == n x (rd_policy_dreamer -> rd_step) bit for bit, deter 36 / hidden 100 / units 132 (a chain
    of 2-CTA clusters) / 3 layers / 360 beams / 257 samples"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n, steps = 300, 20
    w = dp.random_weights(4, n_beams=360, actor_layers=3, deter=36, hidden=100, units=132)
    outs = []
    for mode in ("rollout", "stepwise"):
        env = make_env(n, 360, seed=6, auto_reset=True)
        env.reset()
        pol = DreamerPolicy(env, w, noise="philox", n_samples=257)
        if mode == "rollout":
            pol.rollout(steps)
        else:
            for _ in range(steps):
                env.step(pol.act())
        torch.cuda.synchronize()
        outs.append((env.buf["pose"].clone(), env.buf["lidar"].clone(), pol.actions.clone()) + tuple(t.clone() for t in pol.get_state()))
        env.close()
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    assert np.isfinite(outs[0][0].cpu().numpy()).all()


def test_chain_more_row_blocks_than_resident_clusters(torch_cuda, monkeypatch):
    """units 516: clusters of five CTAs, 5000 envs = 40 row blocks, more than fit the GPU at once -- chain == per-layer
    launches bit for bit, and the actor head against the float64 oracle"""
    torch = torch_cuda
    from racing_dreamer_b200 import DreamerPolicy
    n, S = 5000, 100
    deter, hidden, units, embed, layers = 100, 100, 516, 100, 5
    w = dp.random_weights(8, n_beams=embed, actor_layers=layers, deter=deter, hidden=hidden, units=units)
    env = make_env(n, embed)
    rng = np.random.RandomState(8)
    scan, lidar = scans_of(rng, n, embed, False)
    state = random_state(rng, n, deter)
    es, ea = f32(rng.standard_normal((n, 30))), f32(rng.standard_normal((n, S, 2)))
    outs = []
    for chain in ("1", "0"):
        monkeypatch.setenv("RD_DREAMER_CHAIN", chain)
        pol = DreamerPolicy(env, w, noise="explicit", n_samples=S)
        outs.append(explicit_step(torch, pol, lidar, state, es, ea))
    same_bits(torch, outs[0], outs[1], "chain vs per-layer launches")
    _, _, ref = dp.policy_step(w, scan, tuple(s.astype(np.float64) for s in state), es, ea, np.float64)
    rtol, atol, head = BARS["tf32x3"]
    f = bar_factors(deter, hidden, units, embed, "tf32x3")[2]
    dbg = outs[0][1].cpu().numpy()[n * 60:].reshape(n, 8)
    close("actor_mean", dbg[:, 0:2], ref["actor_mean"], rtol * head * f, atol * head * f, dp.MEAN_SCALE)
    close("actor_std", dbg[:, 2:4], ref["actor_std"], rtol * head * f, atol * head * f, dp.MEAN_SCALE)
    env.close()


def test_rejected_architectures_leave_the_policy_working(torch_cuda):
    """widths that are not multiples of 4, 0 or 8 trunk layers, n_samples 0, embed != n_beams, a device pointer among
    the weights: each raises (in DreamerPolicy or in rd_policy_dreamer_init), and the policy already on the env computes
    what it did before"""
    torch = torch_cuda
    import ctypes as C
    from racing_dreamer_b200 import DreamerPolicy
    n, E = 129, 100
    w = dp.random_weights(2, n_beams=E, actor_layers=3, deter=36, hidden=28, units=132)
    env = make_env(n, E)
    rng = np.random.RandomState(2)
    _, lidar = scans_of(rng, n, E, False)
    state = random_state(rng, n, 36)
    es, ea = f32(rng.standard_normal((n, 30))), f32(rng.standard_normal((n, 100, 2)))
    pol = DreamerPolicy(env, w, noise="explicit")
    want = explicit_step(torch, pol, lidar, state, es, ea)
    arch = dict(n_beams=E, actor_layers=3, deter=36, hidden=28, units=132)
    bad = [dict(arch, deter=38), dict(arch, hidden=30), dict(arch, units=134)]
    for kw in bad:
        with pytest.raises(RuntimeError, match="unsupported Dreamer architecture"):
            DreamerPolicy(env, dp.random_weights(3, **kw), noise="explicit")
    with pytest.raises(ValueError):
        DreamerPolicy(env, {k: v for k, v in w.items() if not (k.startswith("h") and k[1].isdigit())})   # 0 layers
    with pytest.raises(ValueError):
        DreamerPolicy(env, dp.random_weights(3, **dict(arch, actor_layers=8)))
    with pytest.raises(RuntimeError, match="unsupported Dreamer architecture"):
        DreamerPolicy(env, w, n_samples=0)
    with pytest.raises(ValueError):
        DreamerPolicy(env, dp.random_weights(3, **dict(arch, n_beams=96)))
    env98 = make_env(8, 98)
    with pytest.raises(RuntimeError, match="unsupported Dreamer architecture"):
        DreamerPolicy(env98, dp.random_weights(3, **dict(arch, n_beams=98)))   # embed == n_beams, not a multiple of 4
    env98.close()
    # the C ABI's own checks, past DreamerPolicy's
    for field, value in (("actor_layers", 0), ("actor_layers", 8), ("n_samples", 0), ("embed", 96), ("deter", 38),
                         ("actor_units", 130), ("stoch", 32)):
        s = pol._weights_struct(w, None, lambda a: a.ctypes.data_as(C.c_void_p))
        setattr(s, field, value)
        assert env.lib.rd_policy_dreamer_init(env._handle, C.byref(s)) != 0, field
    # init reads host memory: a CUDA tensor's pointer among the weights is rejected, not read on the host
    s = pol._weights_struct(w, None, lambda a: a.ctypes.data_as(C.c_void_p))
    obs2_dev = torch.from_numpy(w["obs2_w"]).cuda()
    s.obs2_w = obs2_dev.data_ptr()
    assert env.lib.rd_policy_dreamer_init(env._handle, C.byref(s)) != 0
    same_bits(torch, explicit_step(torch, pol, lidar, state, es, ea), want, "after the rejected inits")
    env.close()
