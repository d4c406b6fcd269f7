"""CPU checks of the Dreamer-agent oracle (oracle/dreamer_policy.py, SURVEY §8-f2): the checkpoint layout, the GRU cell
against torch.nn.GRUCell (the same published equations with another gate order), the committed golden trajectory, and
SampleDist.mode()'s argmax rule.  The reference's own agent needs TensorFlow, which is not installable here (the
oracle's header says "parity unpinned"); what CAN be pinned is pinned here."""
import numpy as np
import pytest

from oracle import dreamer_policy as dp
from racing_dreamer_b200.policy import load_dreamer_checkpoint, save_dreamer_checkpoint


@pytest.fixture(scope="module")
def weights():
    return load_dreamer_checkpoint("austria_dreamer")


def test_packaged_checkpoint_layout(weights):
    w = weights
    # shapes the reference builds: RSSM(stoch=30, deter=200, hidden=200), ActionDecoder(size=2, layers=4, units=400)
    # [REF ros_agent/models/dreamer/racing_dreamer.py:20-24]; 1080 beams + deter feed obs1 [REF models.py:66-67]
    assert w["gru_kernel"].shape == (200, 600) and w["gru_recurrent"].shape == (200, 600) and w["gru_bias"].shape == (2, 600)
    assert w["img1_w"].shape == (32, 200) and w["obs1_w"].shape == (1280, 200) and w["obs2_w"].shape == (200, 60)
    assert [w[f"h{i}_w"].shape for i in range(4)] == [(230, 400), (400, 400), (400, 400), (400, 400)]
    assert w["hout_w"].shape == (400, 4) and "bn_gamma" not in w
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in w.values())


def test_checkpoint_roundtrip(tmp_path, weights):
    save_dreamer_checkpoint(tmp_path / "ck.npz", weights)
    w2 = load_dreamer_checkpoint(tmp_path / "ck.npz")
    assert set(w2) == set(weights) and all(np.array_equal(w2[k], weights[k]) for k in weights)


def test_pickle_layout_normalized(tmp_path):
    """the 14-variable actor of the 'normalized' agents: hnorm's variables sit between h3 and hout"""
    import pickle
    w = dp.random_weights(3, normalized=True)
    rssm = [w[k] for k in ("gru_kernel", "gru_recurrent", "gru_bias", "img1_w", "img1_b", "img2_w", "img2_b", "img3_w",
                           "img3_b", "obs1_w", "obs1_b", "obs2_w", "obs2_b")]
    actor = sum([[w[f"h{i}_w"], w[f"h{i}_b"]] for i in range(4)], []) + [w["bn_mean"], w["bn_var"], w["bn_gamma"], w["bn_beta"],
                                                                         w["hout_w"], w["hout_b"]]
    (tmp_path / "ck").mkdir()
    pickle.dump(tuple(rssm), open(tmp_path / "ck" / "rssm.pkl", "wb"))
    pickle.dump(tuple(actor), open(tmp_path / "ck" / "actor.pkl", "wb"))
    for loader in (load_dreamer_checkpoint, dp.load_checkpoint):
        w2 = loader(tmp_path / "ck")
        assert set(w2) == set(w) and all(np.array_equal(w2[k], w[k]) for k in w)


def test_gru_cell_matches_torch(weights):
    """tf.keras GRUCell(reset_after=True) [gates z|r|h] == torch.nn.GRUCell [gates r|z|n] after permuting the blocks:
    both compute n = tanh(W_n x + b_in + r * (U_n h + b_hn)), h' = (1 - z) * n + z * h."""
    import torch
    w = weights
    n = 200
    cell = torch.nn.GRUCell(200, n).double()
    perm = np.r_[n:2 * n, 0:n, 2 * n:3 * n]   # keras z|r|h -> torch r|z|n
    with torch.no_grad():
        cell.weight_ih.copy_(torch.from_numpy(w["gru_kernel"].T[perm].astype(np.float64)))
        cell.weight_hh.copy_(torch.from_numpy(w["gru_recurrent"].T[perm].astype(np.float64)))
        cell.bias_ih.copy_(torch.from_numpy(w["gru_bias"][0][perm].astype(np.float64)))
        cell.bias_hh.copy_(torch.from_numpy(w["gru_bias"][1][perm].astype(np.float64)))
    rng = np.random.RandomState(0)
    x, h = rng.standard_normal((16, 200)), rng.uniform(-1, 1, (16, n))
    ours = dp.gru_cell(w, x, h, np.float64)
    with torch.no_grad():
        theirs = cell(torch.from_numpy(x), torch.from_numpy(h)).numpy()
    assert np.abs(ours - theirs).max() < 1e-12


def test_oracle_reproduces_golden(golden_dir, weights):
    g = np.load(golden_dir / "dreamer_policy_golden.npz")
    state = None
    for t in range(g["scans"].shape[0]):
        act, state, d = dp.policy_step(weights, g["scans"][t], state, g["eps_stoch"][t], g["eps_actor"][t], np.float64)
        assert np.array_equal(d["index"], g["index"][t])
        for k, v in (("mean", d["mean"]), ("std", d["std"]), ("stoch", state[0]), ("deter", state[1]),
                     ("actor_mean", d["actor_mean"]), ("actor_std", d["actor_std"]), ("action", act)):
            assert np.abs(v - g[k][t]).max() < 1e-9, k
    # float32 evaluation (what TensorFlow computes in) stays within 1e-3 of the float64 trajectory
    state = None
    for t in range(g["scans"].shape[0]):
        act, state, d = dp.policy_step(weights, g["scans"][t], state, g["eps_stoch"][t], g["eps_actor"][t], np.float32)
        assert np.abs(state[1] - g["deter"][t]).max() < 1e-3 and np.abs(d["mean"] - g["mean"][t]).max() < 1e-3


def test_preprocess_and_postprocess():
    scan = np.array([[-1.0, 0.0, 7.5, 15.0, 20.0]])
    assert np.allclose(dp.preprocess_lidar(scan), [[-0.5, -0.5, 0.0, 0.5, 0.5]])   # [REF racing_dreamer.py:45-52]
    assert np.allclose(dp.postprocess_action(np.array([-2.0, 0.0])), [0.005, 0.0])  # [REF racing_dreamer.py:54-60]
    assert np.allclose(dp.postprocess_action(np.array([1.0, 1.0])), [1.0, 1.0])


def test_mode_is_first_argmax_of_log_prob():
    rng = np.random.RandomState(1)
    mean, std = rng.uniform(-1, 1, (5, 2)), rng.uniform(0.1, 1, (5, 2))
    eps = rng.standard_normal((5, 100, 2))
    eps[:, 7] = eps[:, 3]                                   # a tie: tf.argmax keeps the first
    act, logp, idx, lp = dp.mode(mean, std, eps)
    u = mean[:, None] + std[:, None] * eps
    # independent evaluation of log N(u; mean, std) - log|d tanh/du|
    ref = (-0.5 * ((u - mean[:, None]) / std[:, None]) ** 2 - np.log(std[:, None]) - 0.5 * np.log(2 * np.pi)
           - np.log1p(-np.tanh(u) ** 2)).sum(-1)
    assert np.abs(ref - lp).max() < 1e-9
    assert np.array_equal(idx, ref.argmax(-1)) and not (idx == 7).any()
    assert np.allclose(act, np.tanh(u[np.arange(5), idx]))
    a0, _, i0, _ = dp.mode(mean, std, None)                 # zero-noise variant
    assert np.allclose(a0, np.tanh(mean)) and (i0 == 0).all()


def _torch_step(w, scan, state, eps_stoch, eps_actor):
    """The agent step restated with torch.nn modules in float64: Linear layers for img1, obs1, obs2, the actor trunk
    and hout, torch.nn.GRUCell (gate blocks permuted as in test_gru_cell_matches_torch), BatchNorm1d in eval mode for
    the 'normalized' head, torch.distributions.Normal for the base log-density and log|d tanh(u)/du| = -2 log cosh(u)
    (torch's TanhTransform clips its softplus at 20, 2e-9 away from the exact value for |u| > 10)."""
    import torch
    import torch.nn.functional as F
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64))   # noqa: E731

    def linear(name_w, name_b):
        k = w[name_w]
        lin = torch.nn.Linear(k.shape[0], k.shape[1]).double()
        with torch.no_grad():
            lin.weight.copy_(t(k.T))
            lin.bias.copy_(t(w[name_b]))
        return lin

    deter_n = w["gru_recurrent"].shape[0]
    cell = torch.nn.GRUCell(w["gru_kernel"].shape[0], deter_n).double()
    perm = np.r_[deter_n:2 * deter_n, 0:deter_n, 2 * deter_n:3 * deter_n]
    with torch.no_grad():
        cell.weight_ih.copy_(t(w["gru_kernel"].T[perm]))
        cell.weight_hh.copy_(t(w["gru_recurrent"].T[perm]))
        cell.bias_ih.copy_(t(w["gru_bias"][0][perm]))
        cell.bias_hh.copy_(t(w["gru_bias"][1][perm]))
    softplus = lambda x: F.softplus(x, threshold=50.0)   # noqa: E731  (log1p(exp(x)) over the whole range used here)
    stoch, deter, action = (t(s) for s in state)
    with torch.no_grad():
        embed = (torch.clamp(t(scan), 0.0, 15.0) / 15.0 - 0.5).float().double()   # the scans are preprocessed in float32
        x = F.elu(linear("img1_w", "img1_b")(torch.cat([stoch, action], -1)))
        deter = cell(x, deter)
        x = F.elu(linear("obs1_w", "obs1_b")(torch.cat([deter, embed], -1)))
        mean, raw = linear("obs2_w", "obs2_b")(x).split(dp.STOCH, -1)
        std = softplus(raw) + 0.1
        stoch = mean + std * t(eps_stoch)
        x = torch.cat([stoch, deter], -1)
        for i in range(dp.n_actor_layers(w)):
            x = F.elu(linear(f"h{i}_w", f"h{i}_b")(x))
        x = linear("hout_w", "hout_b")(x)
        if "bn_gamma" in w:
            bn = torch.nn.BatchNorm1d(4, eps=dp.BN_EPS).double().eval()
            bn.weight.copy_(t(w["bn_gamma"]))
            bn.bias.copy_(t(w["bn_beta"]))
            bn.running_mean.copy_(t(w["bn_mean"]))
            bn.running_var.copy_(t(w["bn_var"]))
            x = bn(x)
            amean, astd = x[:, :2], softplus(x[:, 2:]) + dp.MIN_STD
        else:
            amean = dp.MEAN_SCALE * torch.tanh(x[:, :2] / dp.MEAN_SCALE)
            astd = softplus(x[:, 2:] + float(np.log(np.exp(dp.INIT_STD) - 1))) + dp.MIN_STD
        u = amean[:, None] + astd[:, None] * t(eps_actor)
        lp = (torch.distributions.Normal(amean[:, None], astd[:, None]).log_prob(u) + 2.0 * torch.log(torch.cosh(u))).sum(-1)
    return {k: v.numpy() for k, v in dict(mean=mean, std=std, stoch=stoch, deter=deter, actor_mean=amean,
                                          actor_std=astd, logp_all=lp).items()}


@pytest.mark.parametrize("deter,hidden,units,embed,layers,normalized", [
    (36, 100, 132, 100, 3, False), (4, 4, 4, 4, 1, False), (212, 28, 32, 360, 5, True), (516, 1028, 1028, 2048, 2, False)])
def test_oracle_matches_torch_at_other_architectures(deter, hidden, units, embed, layers, normalized):
    """The oracle generalised to any width (random_weights, policy_step) == an independent torch.nn restatement to
    1e-12: what makes it the yardstick of the kernels at architectures other than the shipped one."""
    w = dp.random_weights(7, n_beams=embed, normalized=normalized, actor_layers=layers, deter=deter, hidden=hidden, units=units)
    assert w["gru_recurrent"].shape == (deter, 3 * deter) and w["obs1_w"].shape == (deter + embed, hidden)
    assert dp.n_actor_layers(w) == layers and w["hout_w"].shape == (units, 4) and w[f"h{layers - 1}_w"].shape[1] == units
    rng = np.random.RandomState(1)
    n, S = 24, 37
    scan = rng.uniform(-1, 18, (n, embed))
    state = (rng.standard_normal((n, 30)), rng.uniform(-1, 1, (n, deter)), rng.uniform(-1, 1, (n, 2)))
    es, ea = rng.standard_normal((n, 30)), rng.standard_normal((n, S, 2))
    act, new_state, d = dp.policy_step(w, scan, state, es, ea, np.float64)
    ref = _torch_step(w, scan, state, es, ea)
    got = dict(mean=d["mean"], std=d["std"], stoch=new_state[0], deter=new_state[1], actor_mean=d["actor_mean"],
               actor_std=d["actor_std"], logp_all=d["logp_all"])
    for k, v in got.items():
        assert v.shape == ref[k].shape and np.abs(v - ref[k]).max() <= 1e-12 * max(1.0, np.abs(ref[k]).max()), k
    assert np.array_equal(d["index"], ref["logp_all"].argmax(-1))
    # the zero state is as wide as the weights' GRU
    _, s0, _ = dp.policy_step(w, scan, None, es, ea, np.float64)
    assert s0[1].shape == (n, deter)


def test_random_weights_defaults_unchanged():
    """the generalised random_weights draws the shipped architecture's arrays exactly as before (the goldens and the
    GPU tests' weights depend on them): the default widths given explicitly change nothing"""
    a = dp.random_weights(11, normalized=True)
    b = dp.random_weights(11, n_beams=1080, normalized=True, actor_layers=4, deter=200, hidden=200, units=400)
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert a["gru_kernel"].shape == (200, 600) and a["h3_w"].shape == (400, 400) and a["obs1_w"].shape == (1280, 200)
