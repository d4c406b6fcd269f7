"""CPU: the oracle against the fixtures recorded from the UNMODIFIED reference classes (tests/golden/make_golden.py)."""
import numpy as np
import pytest

import helpers
from oracle import Oracle, default_config, ref_stubs
from racing_dreamer_b200 import _abi, load_track


def test_occupancy_matches_reference_class(golden_dir):
    """a5: OccupancyMapObs.step [REF dreamer/wrappers.py:390-408] -- bit-exact on every golden pose."""
    g = np.load(golden_dir / "occupancy_golden.npz")
    names = [str(n) for n in g["track_names"]]
    cfg = default_config()
    orc = Oracle(cfg, [load_track(n) for n in names], n_threads=4)
    got = orc.occupancy_obs(g["poses"], g["track"])
    want = np.unpackbits(g["images"], axis=2)[:, :, :64]
    assert got.shape == want.shape
    assert np.array_equal(got, want)
    assert set(np.unique(got)) <= {0, 1}


def test_dreamer_stack_replay(golden_dir):
    """a3,a4,a9,a10,a11: fused step == RaceCarWrapper/ActionRepeat/ReduceActionSpace/OccupancyMapObs/TimeLimit/Collect
    of the reference [REF dreamer/wrappers.py:22-250] run tick by tick (BASELINE config 1)."""
    g = np.load(golden_dir / "dreamer_stack_golden.npz")
    cfg = helpers.fused_dreamer_config(default_config(), int(g["action_repeat"]), int(g["duration"]))
    orc = Oracle(cfg, [load_track("columbia")])
    rec = helpers.replay(lambda: orc.reset(mode=_abi.RESET_GRID), lambda a: orc.step(a), g["actions"], g["reset_before"])
    helpers.assert_matches_dreamer_golden(rec, g)


def test_baselines_stack_replay(golden_dir):
    """a4,a9 (baselines variants): Flatten clip + ActionRepeat that does not test the first tick's done
    [REF baselines/racing/environment/single_agent.py:31-62]."""
    g = np.load(golden_dir / "baselines_stack_golden.npz")
    cfg = helpers.fused_baselines_config(default_config(), int(g["repeat"]))
    orc = Oracle(cfg, [load_track("austria")])
    rec = helpers.replay(lambda: orc.reset(mode=_abi.RESET_GRID), lambda a: orc.step(a), g["actions"], g["reset_before"])
    helpers.assert_matches_baselines_golden(rec, g)


def test_library_stages_against_scipy_and_pillow():
    """The two library stages of a5, restated in the oracle, against the libraries themselves."""
    from PIL import Image
    from scipy import ndimage
    rng = np.random.RandomState(3)
    a = (rng.rand(220, 220) > 0.5).astype(np.uint8)
    ref = ndimage.spline_filter(a, order=3, output=np.float64, mode="constant")
    assert np.abs(ref - Oracle.spline_prefilter_2d(a.astype(np.float64))).max() < 1e-13
    for trial in range(4):
        b = (rng.rand(200, 200) > rng.uniform(0.2, 0.8)).astype(np.uint8)
        assert np.array_equal(np.array(Image.fromarray(b).resize((64, 64))), Oracle.pil_resize_200_to_64(b))


@pytest.mark.skipif(not ref_stubs.available(), reason="/root/reference not present (GPU box)")
def test_reference_wrapper_arithmetic_live():
    """a4/a11 on fresh inputs, straight from the reference's classes (not via fixtures)."""
    W = ref_stubs.reference_wrappers()

    class Dummy:
        agent_ids = ["A"]

        def step(self, a):
            self.last = a
            return {}, {}, {}, {}

    d = Dummy()
    r = W.ReduceActionSpace(d, low=[0.005, -1.0], high=[1.0, 1.0])
    rng = np.random.RandomState(0)
    acts = rng.uniform(-1, 1, (64, 2)).astype(np.float32)
    cfg = default_config()
    for a in acts:
        r.step({"A": a})
        t = (a + np.float32(1.0)) / np.float32(2.0)
        mine = t.astype(np.float64) * (np.array([1.0, 1.0]) - np.array([0.005, -1.0])) + np.array([0.005, -1.0])
        assert np.array_equal(d.last["A"], mine)
    assert cfg.action_low[0] == 0.005 and cfg.action_high[0] == 1.0


@pytest.mark.parametrize("name", ["train", "test"])
def test_baselines_chain_replay(golden_dir, name):
    """a11 + the model-free chain end to end: FilterObservation(['lidar']) -> Flatten -> NormalizeObservations
    (-> InfoToObservation) -> FixedResetMode -> gym TimeLimit (ticks, inside ActionRepeat) -> ActionRepeat of the
    reference [REF baselines/racing/experiments/acme/experiment.py:66-88; baselines/racing/environment/
    single_agent.py:31-99; common.py:22-39] == one fused step with RD_OBS_NORM_BASELINES + time_limit_ticks."""
    g = np.load(golden_dir / "baselines_chain_golden.npz")
    cfg = helpers.fused_baselines_chain_config(default_config(), g, test=(name == "test"))
    orc = Oracle(cfg, [load_track("treitlstrasse_v2")])
    rec = helpers.replay(lambda: orc.reset(mode=_abi.RESET_GRID), lambda a: orc.step(a), g["actions"],
                         g[f"{name}_reset_before"])
    helpers.assert_matches_baselines_chain_golden(rec, g, name)
    assert g[f"{name}_truncated"].sum() > 0                      # the tick limit really fired in the recording


def test_simulate_statistics(golden_dir):
    """a12: the per-episode statistics of the reference's driver loop tools.simulate [REF dreamer/tools.py:154-206]
    (max over the episode of lap + progress - 1, cumulative reward of the first agent) from the device-side accumulators'
    CPU restatement."""
    g = np.load(golden_dir / "simulate_golden.npz")
    cfg = helpers.fused_dreamer_config(default_config(), int(g["action_repeat"]), int(g["duration"]), occupancy=False)
    orc = Oracle(cfg, [load_track("treitlstrasse_v2")])
    returns, maxima = helpers.simulate_statistics(lambda: orc.reset(mode=_abi.RESET_GRID), lambda a: orc.step(a),
                                                  lambda: orc.read_stats(reset=True), g)
    assert np.allclose(returns, g["cum_rewards"], rtol=1e-12, atol=1e-12)
    assert np.allclose(maxima, g["max_progresses"], rtol=0, atol=1e-12)
