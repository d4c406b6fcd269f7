"""CPU: compiled tracks (a6) -- format, geometry conventions, and the generator restatement."""
import numpy as np
import pytest

from racing_dreamer_b200 import TRACK_FILES, load_track, maps

# lap lengths of the paper's tracks (SURVEY.md Appendix B): wavefront distance * 0.05 m
LAP_M = {"austria": 79.45, "barcelona": 201.0, "treitlstrasse_v2": 51.65, "columbia": 61.2, "circle_cw": 41.9}


@pytest.mark.parametrize("name", sorted(TRACK_FILES))
def test_compiled_track(name):
    tm = load_track(name)
    assert tm.resolution == 0.05 and tm.full_shape == (2000, 2000)
    if name in LAP_M:
        assert abs(tm.lap_length_m() - LAP_M[name]) < 0.051
    d = tm.drivable
    assert not d[:maps.MARGIN].any() and not d[-maps.MARGIN:].any() and not d[:, :maps.MARGIN].any() and not d[:, -maps.MARGIN:].any()
    assert tm.dist.max() == tm.dmax and (tm.dist[~d] == 0).all()
    bits = tm.packed_bits_yup()
    assert bits.shape == (tm.h, tm.row_words()) and tm.row_words() % 2 == 1
    un = ((bits[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(tm.h, -1)[:, :tm.w].astype(bool)
    assert np.array_equal(un, d[::-1])
    # start pixel = world (0,0) -> (row 999, col 1000) [REF docs/maps/costmaps/generate-costmap.py:49-52]
    assert tm.to_pixel(0.0, 0.0) == (999, 1000)
    r, c = tm.to_pixel(*tm.start_poses[0, :2])
    assert d[r - tm.r0, c - tm.c0] and tm.dist[r - tm.r0, c - tm.c0] == 0
    # every reset pose sits on a drivable cell with clearance
    for x, y, _ in tm.reset_poses[:: max(1, len(tm.reset_poses) // 64)]:
        r, c = tm.to_pixel(x, y)
        assert d[r - tm.r0, c - tm.c0] and tm.edt_sq[r - tm.r0, c - tm.c0] >= 64


def test_reference_format_arrays():
    tm = load_track("treitlstrasse_v2")
    full = tm.full_drivable()
    assert full.shape == (2000, 2000) and full.sum() == tm.drivable.sum()
    nd = tm.full_norm_distance_from_start()
    assert nd.max() == 1.0 and nd.min() == 0.0
    no = tm.full_norm_distance_to_obstacle()
    assert no.max() == 1.0 and (no[~full] == 0).all()


@pytest.fixture(scope="module")
def map_dir(tmp_path_factory):
    """map_server sources (yaml + 1-bit png) of the tracks the compiler tests read.  The compilers use an image only
    through its free area connected to the start pixel, so an image whose free cells are a shipped track's drivable
    area compiles exactly as the original map does; the generator fixtures compared against below were recorded from
    the original map images."""
    from PIL import Image
    d = tmp_path_factory.mktemp("maps")
    for name in ("treitlstrasse_v2", "austria", "columbia"):
        tm, stem = load_track(name), TRACK_FILES[name]
        Image.fromarray(tm.full_drivable()).save(d / f"{stem}.png")
        (d / f"{stem}.yaml").write_text(f"image: {stem}.png\nresolution: {tm.resolution}\n"
                                        f"origin: [{tm.origin[0]}, {tm.origin[1]}, 0.0]\noccupied_thresh: 0.65\n")
    return d


def test_recompile_matches_stored_and_dilation_wavefront(map_dir):
    """Recompiling from the map source reproduces the stored npz, and the frontier BFS equals the
    generator's literal repeated-3x3-dilation wavefront [REF docs/maps/costmaps/generate-costmap.py:198-209]."""
    from scipy import ndimage
    tm = load_track("treitlstrasse_v2")
    fresh = maps.compile_track(map_dir / "Treitlstrasse_3-U_v2.yaml")
    assert np.array_equal(fresh.drivable, tm.drivable) and np.array_equal(fresh.dist, tm.dist)
    assert np.array_equal(fresh.reset_poses, tm.reset_poses)
    free = tm.drivable & (tm.dist < tm.dmax)
    r, c = tm.to_pixel(0.0, 0.0)
    mask = np.zeros_like(free)
    mask[r - tm.r0, c - tm.c0] = True
    dist = np.zeros(free.shape, np.int32)
    cur = 0
    while True:
        cur += 1
        new = free & (ndimage.binary_dilation(mask, structure=np.ones((3, 3), bool)) ^ mask)
        if not new.any():
            break
        dist[new] = cur
        mask |= new
    assert cur == tm.dmax
    assert np.array_equal(dist[free], tm.dist[free].astype(np.int32))


# ---------------------------------------------------------------------------------------------------------
# a6 / §8-f4: pinned against the UNMODIFIED generator (tests/golden/costmap_golden.npz, oracle/ref_costmap.py)
def _golden_layers(golden_dir, name):
    g = np.load(golden_dir / "costmap_golden.npz")
    r0, c0, h, w = (int(v) for v in g[f"{name}_r0c0hw"])
    drv = np.unpackbits(g[f"{name}_drivable"], axis=1)[:, :w].astype(bool)
    return (r0, c0, h, w), drv, g[f"{name}_dist"], int(g[f"{name}_dmax"]), g[f"{name}_edt_sq"]


def test_shipped_austria_equals_reference_generator(golden_dir):
    """f1_aut: the generator's cleared pixel is off the track, so the shipped track IS the generator's output"""
    (r0, c0, h, w), drv, dist, dmax, edt = _golden_layers(golden_dir, "austria")
    tm = load_track("austria")
    assert (tm.r0, tm.c0, tm.h, tm.w, tm.dmax) == (r0, c0, h, w, dmax)
    assert np.array_equal(tm.drivable, drv) and np.array_equal(tm.dist, dist) and np.array_equal(tm.edt_sq, edt)


def test_shipped_treitlstrasse_differs_only_by_the_cleared_pixel(golden_dir):
    """Treitlstrasse_3-U_v2: the generator clears pixel (987, 1294) of every map [REF generate-costmap.py:45-46]; it is
    on this track.  The shipped track keeps it drivable (no phantom 5 cm wall for the ray caster); everything else is
    the generator's output, up to the detour the wavefront takes around the hole."""
    (r0, c0, h, w), drv, dist, dmax, edt = _golden_layers(golden_dir, "treitlstrasse_v2")
    tm = load_track("treitlstrasse_v2")
    assert (tm.r0, tm.c0, tm.h, tm.w, tm.dmax) == (r0, c0, h, w, dmax)
    pr, pc = maps.REFERENCE_CLEARED_PIXEL[0] - r0, maps.REFERENCE_CLEARED_PIXEL[1] - c0
    diff = np.argwhere(tm.drivable != drv)
    assert diff.tolist() == [[pr, pc]] and tm.drivable[pr, pc] and not drv[pr, pc]
    rr, cc = np.mgrid[0:h, 0:w]
    far = np.maximum(np.abs(rr - pr), np.abs(cc - pc)) > 40
    dd = np.abs(tm.dist.astype(np.int64) - dist.astype(np.int64))
    assert dd[far].max() == 0 and dd[(~far) & drv].max() <= 1        # one-cell detour right behind the hole
    assert np.array_equal(tm.edt_sq[far], edt[far])


def test_compile_with_reference_quirks_reproduces_golden(golden_dir, map_dir):
    """compile_track(reference_quirks=True) == the generator's arrays, bit for bit (fixture made by running the
    unmodified script; see tests/golden/make_golden.py::costmap_golden)"""
    for name in ("treitlstrasse_v2", "austria"):
        (r0, c0, h, w), drv, dist, dmax, edt = _golden_layers(golden_dir, name)
        tm = maps.compile_track(map_dir / f"{TRACK_FILES[name]}.yaml", reference_quirks=True)
        assert (tm.r0, tm.c0, tm.h, tm.w, tm.dmax) == (r0, c0, h, w, dmax)
        assert np.array_equal(tm.drivable, drv) and np.array_equal(tm.dist, dist) and np.array_equal(tm.edt_sq, edt)


def test_distance_to_target_layer_reproduces_generator(golden_dir, map_dir):
    """§8-f4: the generator's fourth stored layer, `norm_distance_to` (smoothed distance to the target)
    [REF docs/maps/costmaps/generate-costmap.py:227-276,405-420], restated in maps.compile_distance_to_target; the fixture
    is the unmodified script's full run() on Treitlstrasse_3-U_v2 (tests/golden/make_golden.py::costmap_golden)."""
    import hashlib
    g = np.load(golden_dir / "costmap_golden.npz")
    out = maps.compile_distance_to_target(map_dir / "Treitlstrasse_3-U_v2.yaml", reference_quirks=True)
    ndt = np.ascontiguousarray(out["norm_distance_to"], dtype=np.float64)
    r0, c0, h, w = (int(v) for v in g["treitlstrasse_v2_r0c0hw"])
    assert np.abs(ndt[r0:r0 + h, c0:c0 + w].astype(np.float32) - g["treitlstrasse_v2_norm_distance_to_crop_f32"]).max() == 0.0
    assert hashlib.sha256(ndt.tobytes()).hexdigest() == str(g["treitlstrasse_v2_norm_distance_to_sha256"])
    assert ndt.max() == 1.0 and (ndt[~out["drivable_area"]] == 0).all()
    # maps with custom generator settings keep the plain wavefront distance (use_blurred_factor off) [REF :94-105]
    plain = maps.compile_distance_to_target(map_dir / "f1_aut.yaml")
    d = plain["norm_distance_to"][plain["drivable_area"]]
    steps = np.unique(np.round(d * d.size))          # a pure wavefront distance takes few distinct values per cell count
    assert len(np.unique(d)) <= 2000 and steps.size > 10

@pytest.mark.parametrize("name", ["austria", "columbia"])
def test_raceline_layer_reproduces_generator(golden_dir, map_dir, name):
    """§8-f4: the race-line layer the generator draws on the eroded track [REF docs/maps/costmaps/generate-costmap.py:
    280-360, called at :378], restated in maps.compile_raceline; the fixture is what the UNMODIFIED compute_raceline
    returned inside the script's full run() (tests/golden/make_golden.py::raceline_golden), on the two maps that carry
    their own erosion / spline degree / sampling settings [REF :83-106]."""
    import hashlib
    g = np.load(golden_dir / "raceline_golden.npz")
    out = maps.compile_raceline(map_dir / f"{TRACK_FILES[name]}.yaml", reference_quirks=True)
    layer = np.ascontiguousarray(out["raceline"], dtype=np.float64)
    r0, c0, h, w = (int(v) for v in g[f"{name}_r0c0hw"])
    assert np.array_equal(out["control_points"], g[f"{name}_control_points"])
    assert np.abs(layer[r0:r0 + h, c0:c0 + w].astype(np.float32) - g[f"{name}_crop_f32"]).max() == 0.0
    assert int((layer > 0).sum()) == int(g[f"{name}_nonzero"])
    assert hashlib.sha256(layer.tobytes()).hexdigest() == str(g[f"{name}_sha256"])
    # properties: normalised, confined to the drivable area, a closed loop of control points that stays on the track
    drivable = maps.compile_distance_to_target(map_dir / f"{TRACK_FILES[name]}.yaml",
                                               reference_quirks=True)["drivable_area"]
    assert layer.max() == 1.0 and layer.min() >= 0.0 and (layer[~drivable] == 0).all()
    cp = out["control_points"]
    assert cp.shape[0] > 20 and drivable[cp[:, 0], cp[:, 1]].all()
    assert np.abs(cp[0] - cp[-1]).max() < 60          # the descent comes back to where it started

