"""CPU: the case table, the synthetic inputs and the error bar of the model-free actor's shape tests
(test_gpu_sb3_shapes.py imports them), and a check that the bar has teeth: NumPy emulations of the ways the kernels
could be subtly wrong fail it, the emulation of what they are meant to compute passes it.

What the kernels accept (rd_mlp.cuh mlp_check): 1..4 layers of any width 1..1024, in_features = n_beams any multiple of
4 up to 8192, relu or tanh, a squashed (SAC) or diagonal (PPO / A2C) head.  What the chosen values reach (128-wide N
tiles, 32-wide K blocks, widths padded to multiples of 4 by mlp_pad4, packed by k_pack_weights<KMAJOR> with row pitch
ld = the padded width of the layer before):
  * widths 1, 2, 3 pad to 4: a 4-column N tile, and the next layer's K is one partial block; 5 -> 8, 33 -> 36,
    127 -> 128, 129 -> 132 (two N tiles, the last 4 columns wide), 255 -> 256, 257 -> 260, 1021 / 1023 -> 1024;
  * every width that is not a multiple of 4 makes the next matrix's pitch ld != in (the packer's pitch, zero K slots);
  * 4 / 100 / 360 / 1080 beams: a partial last K block of layer 0; 2048 / 8192: exact blocks, 8192 = 256 blocks in
    dr_build's 3 accumulator groups of ~86 (the shipped 1080-beam layer: 34 blocks, 12 per group);
  * 1024-wide layers: 8 N tiles; 5000 envs: 40 row blocks, more CTAs than fit the device at once;
  * 1, 127, 128, 129, 300 envs: around the 128-row tiles.

The bar.  rd_mlp.cuh claims float32-grade products (tf32x3: hi*hi + hi*lo + lo*hi).  Per quantity q (the Gaussian's
mean and std) and case:  bar_q = max(8 E32_q, ETF_q / 8) + 2^-21 S_q,  E32 = the largest error of a float32 evaluation
of the actor against float64 (x3 products carry ~2^-21 relative error, float32 ones 2^-24), ETF = the largest error of
one TF32 pass (tf32_single below), S = the largest |ref_q| (a few ulp of expf / tanhf).  The kernel must be float32-grade
and at least 8x better than one TF32 pass.  Actions, element by element: |d a| <= bar_mean + |e| bar_std (tanh and the
sample a = mean + std e move by at most that).

Emulations (NumPy, float64 sums): tf32_single -- both operands rounded to TF32 as k_pack_weights rounds (ties away from
zero), one product; x3 -- hi*hi + hi*lo + lo*hi; k_tail_dropped -- the last partial K block of layer 0 read as zeros;
pitch_ignored -- every matrix packed with pitch in and read with pitch ld."""
import zlib

import numpy as np
import pytest

from oracle import sb3_policy as sp
from test_cpu_sb3_policy import make_sd

F32_MULTIPLE = 8.0    # 2^-21 / 2^-24: an x3 product against a float32 one
TF32_DIVISOR = 8.0    # the kernel must beat one TF32 pass by this much
ULP_TERM = 2.0 ** -21
TEETH = 4.0           # tf32_single must miss the bar by at least this factor
GM_BK = 32            # K block (floats)


def case(algo, widths, n_beams, n_envs, activation=None, shared=0, refresh=False, scale=1.0):
    """widths: the whole trunk; for ppo the first `shared` of them are mlp_extractor.shared_net"""
    return dict(algo=algo, widths=tuple(widths), n_beams=n_beams, n_envs=n_envs,
                activation=activation or ("relu" if algo == "sac" else "tanh"), shared=shared, refresh=refresh,
                scale=scale)


# hand-picked: each names the path it reaches (module docstring)
CASES = {
    "width1":          case("sac", [1], 1080, 129, refresh=True),                     # head packer ld 4 != in 1
    "widths3_5_tanh":  case("sac", [3, 5], 100, 127, "tanh"),                          # 1-wide partial K block, K tail
    "beams4_relu_ppo": case("ppo", [33], 4, 1, "relu"),                                # a single 4-wide K block, one row
    "tile_tails":      case("ppo", [129, 127, 255, 2], 1080, 300, shared=1, refresh=True),   # 132 = 128 + 4 columns
    "max_width":       case("sac", [1024] * 4, 2048, 128, refresh=True),              # 8 N tiles, 64 exact K blocks
    "max_beams":       case("sac", [1021, 1023], 8192, 300, refresh=True),            # 256 K blocks, 86 per group
    "bottleneck":      case("ppo", [1024, 1, 1024], 360, 129),                        # K = 4 between two widest layers
    "many_row_blocks": case("sac", [1024, 255], 1080, 5000),                          # 40 row blocks x 8 N tiles
    "saturated_tanh":  case("ppo", [64, 64], 1080, 300, scale=8.0),                   # tanh saturated in the epilogue
    "large_relu":      case("sac", [256, 256], 1080, 300, scale=4.0),                 # dead units, large activations
}
SWEEP_WIDTHS = [1, 2, 3, 5, 33, 127, 129, 255, 257, 1021, 1024]
N_SWEEP = 12


def sweep_case(seed):
    r = np.random.RandomState(7000 + seed)
    algo = str(r.choice(["sac", "ppo"]))
    widths = [int(r.choice(SWEEP_WIDTHS)) for _ in range(int(r.randint(1, 5)))]
    shared = int(algo == "ppo" and len(widths) > 1 and r.rand() < 0.5)
    return case(algo, widths, int(r.choice([4, 100, 1080, 2048])), int(r.choice([1, 127, 128, 129, 300])),
                str(r.choice(["relu", "tanh"])), shared, refresh=bool(r.rand() < 0.25))


ALL_CASES = {**CASES, **{f"sweep{s}": sweep_case(s) for s in range(N_SWEEP)}}


def case_seed(name):
    return zlib.crc32(name.encode()) % 100000


def case_sd(c, seed, **kw):
    """the case's SB3 state dict (weights from `seed`)"""
    w = c["widths"]
    if c["algo"] == "sac":
        return make_sd("sac", seed, c["n_beams"], widths=w, scale=c["scale"], **kw)
    return make_sd("ppo", seed, c["n_beams"], widths=w[c["shared"]:], shared=w[:c["shared"]], scale=c["scale"], **kw)


def case_weights(c, seed, **kw):
    """(state dict, canonical weights) of the case"""
    from racing_dreamer_b200.policy import load_sb3_checkpoint
    sd = case_sd(c, seed, **kw)
    return sd, load_sb3_checkpoint(sd, activation=c["activation"], n_beams=c["n_beams"])[1]


def synthetic_scans(seed, n, n_beams):
    """float32 scans as the baselines chain normalises them: uniform in [0, 1], the first row all zeros and the last
    all ones (when there are at least three rows)"""
    x = np.random.default_rng(seed).uniform(0.0, 1.0, (n, n_beams)).astype(np.float32)
    if n >= 3:
        x[0], x[-1] = 0.0, 1.0
    return x


# --- emulations of the products ------------------------------------------------------------------------------------
def tf32(x):
    """k_pack_weights' rounding to TF32 (gm_tf32_bits: ties away from zero on the bits; cvt.rna for the scans)"""
    b = np.ascontiguousarray(x, np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def split(x):
    x = np.asarray(x, np.float32)
    h = tf32(x)
    return h.astype(np.float64), tf32(x - h).astype(np.float64)


def mm_tf32_single(a, w):
    """one TF32 pass: both operands' hi, products summed in float64"""
    return split(a)[0] @ split(w)[0].T


def mm_x3(a, w):
    """what the kernels compute: hi*hi + hi*lo + lo*hi (float32 operands: the epilogue stores float32 activations)"""
    (ah, al), (wh, wl) = split(a), split(w)
    return ah @ wh.T + ah @ wl.T + al @ wh.T


def k_tail_dropped(obs):
    k = obs.shape[1] // GM_BK * GM_BK
    out = np.array(obs)
    out[:, k:] = 0.0
    return out


def pitch_ignored(w):
    """each matrix [out][in] packed as if its row pitch were in, read with pitch ld = in rounded up to 4"""
    out = dict(w)
    for k, m in w.items():
        if m.ndim == 2 and m.shape[1] % 4:
            o, i = m.shape
            flat = np.zeros(o * ((i + 3) // 4 * 4), np.float32)
            flat[:o * i] = m.ravel()
            out[k] = flat.reshape(o, -1)[:, :i].copy()
    return out


# --- the bar --------------------------------------------------------------------------------------------------------
def reference(w, c, obs, eps=None, log_std_bounds=(sp.LOG_STD_MIN, sp.LOG_STD_MAX)):
    """float64 (mean, std, action) of the case and the bars {mean, std} of the module docstring"""
    run = lambda **kw: sp.actor(w, c["algo"], c["activation"], obs, eps, eps is None, log_std_bounds=log_std_bounds,   # noqa: E731
                                **kw)
    ref = run()
    e32 = [np.abs(np.float64(x) - r).max() for x, r in zip(run(dtype=np.float32), ref)]
    etf = [np.abs(x - r).max() for x, r in zip(run(matmul=mm_tf32_single), ref)]
    bars = {q: max(F32_MULTIPLE * e32[i], etf[i] / TF32_DIVISOR) + ULP_TERM * np.abs(ref[i]).max()
            for i, q in enumerate(("mean", "std"))}
    return ref, bars


def worst_over_bar(got, ref, bars, eps=None):
    """{mean, std, action: the largest |got - ref| / bar}; got, ref: (mean, std, action)"""
    out = {}
    for i, q in enumerate(("mean", "std")):
        out[q] = float(np.abs(np.float64(got[i]) - ref[i]).max() / bars[q])
    e = 0.0 if eps is None else np.abs(np.float64(eps))
    out["action"] = float((np.abs(np.float64(got[2]) - ref[2]) / (bars["mean"] + e * bars["std"])).max())
    return out


def check(what, got, ref, bars, eps=None):
    """got (mean, std, action) within the bars; returns worst_over_bar"""
    r = worst_over_bar(got, ref, bars, eps)
    assert max(r.values()) <= 1.0, f"{what}: |err| / bar {r} (bars {bars})"
    return r


@pytest.mark.parametrize("name", list(ALL_CASES))
def test_bar_has_teeth(name):
    c = ALL_CASES[name]
    seed = case_seed(name)
    _, w = case_weights(c, seed)
    obs = synthetic_scans(seed, c["n_envs"], c["n_beams"])
    ref, bars = reference(w, c, obs)
    act = lambda ww, x, **kw: sp.actor(ww, c["algo"], c["activation"], x, **kw)   # noqa: E731
    ratios = {"x3": worst_over_bar(act(w, obs, matmul=mm_x3), ref, bars),
              "tf32_single": worst_over_bar(act(w, obs, matmul=mm_tf32_single), ref, bars)}
    assert max(ratios["x3"].values()) <= 0.01, ratios["x3"]
    assert ratios["tf32_single"]["mean"] >= TEETH, ratios["tf32_single"]
    if c["algo"] == "sac":
        assert ratios["tf32_single"]["std"] >= TEETH, ratios["tf32_single"]
    if c["n_beams"] % GM_BK:
        ratios["k_tail_dropped"] = worst_over_bar(act(w, k_tail_dropped(obs), matmul=mm_x3), ref, bars)
        assert max(ratios["k_tail_dropped"].values()) > 1.0, ratios["k_tail_dropped"]
    if any(u % 4 for u in c["widths"]):
        ratios["pitch_ignored"] = worst_over_bar(act(pitch_ignored(w), obs, matmul=mm_x3), ref, bars)
        assert max(ratios["pitch_ignored"].values()) > 1.0, ratios["pitch_ignored"]
    print(name, c["algo"], c["activation"], c["widths"], c["n_beams"], c["n_envs"], "|err| / bar:",
          {k: {q: f"{v:.3g}" for q, v in r.items()} for k, r in ratios.items()})


def test_emulations():
    """the TF32 rounding is k_pack_weights' (ties away from zero), hi + lo is x to 2^-22, pitch_ignored is the packer's
    index f = (e / in) ld + e % in read back with pitch ld"""
    x = np.float32([1.0 + 2.0 ** -11, -(1.0 + 2.0 ** -11), 1.0 + 2.0 ** -12, 1.0 + 3 * 2.0 ** -11, 0.0])
    np.testing.assert_array_equal(tf32(x), np.float32([1.0 + 2.0 ** -10, -(1.0 + 2.0 ** -10), 1.0, 1.0 + 2.0 ** -9, 0.0]))
    v = np.random.default_rng(0).standard_normal(1000).astype(np.float32)
    h, lo = split(v)
    assert np.all(np.abs(h + lo - v) <= 2.0 ** -22 * np.abs(v)) and np.all(tf32(v) == np.float32(h))
    m = np.arange(1, 7, dtype=np.float32).reshape(2, 3)
    np.testing.assert_array_equal(pitch_ignored({"w": m})["w"], np.float32([[1, 2, 3], [5, 6, 0]]))
    np.testing.assert_array_equal(k_tail_dropped(np.ones((1, 40)))[0], [1.0] * 32 + [0.0] * 8)


def test_scale_and_float32_evaluation():
    """scale multiplies the trunk only; the float32 evaluation is float32 throughout and close to float64"""
    a, b = sp.sac_state_dict(3, 100, widths=(8,)), sp.sac_state_dict(3, 100, widths=(8,), scale=4.0)
    for k in a:
        np.testing.assert_allclose(b[k], a[k] * (4.0 if k.startswith("actor.latent_pi") else 1.0), rtol=1e-6)
    c = case("ppo", [8, 8], 100, 5, shared=1)
    sd = case_sd(c, 1, log_std=(0.5, 0.5))
    assert sd["mlp_extractor.shared_net.0.weight"].shape == (8, 100) and sd["log_std"][0] == np.float32(0.5)
    _, w = case_weights(CASES["large_relu"], 2)
    obs = synthetic_scans(2, 9, 1080)
    r32 = sp.actor(w, "sac", "relu", obs, dtype=np.float32)
    r64 = sp.actor(w, "sac", "relu", obs)
    assert all(x.dtype == np.float32 for x in r32)
    assert all(np.abs(x - y).max() < 1e-4 for x, y in zip(r32, r64))
