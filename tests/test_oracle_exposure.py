"""Exposure compensation (include/mcs.h mcs_plan_estimate_gains / mcs_plan_set_exposure_gains), CPU side: the
restatement ``oracle/exposure_model.py`` against OpenCV's GainCompensator.

- ``stats`` and ``cv2.solve`` give ``getMatGains()`` bit for bit on seeded sets of 2-8 random rectangles with
  per-camera brightness scales and masks of 0, partial values and 255; on contained and disjoint rectangles, overlaps
  without a common 255 pixel (N = 1), all cameras isolated (every gain 1) and the 28 random rigs under every map kind;
- ``solve`` (the library's elimination) is within 1e-12 relative of ``cv2.solve`` and gives the same 256-entry tables;
- ``apply`` equals cv2's ``apply`` on all 256 values, for 1, 3 and 4 channels;
- ``blend_*`` equals ``blend_*_cv2``;
- the Python entry points validate their input without a GPU."""
import pickle

import cv2
import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, chain_case, make_maps
from multicamera_stitching_b200 import Stitcher
from multicamera_stitching_b200.plan import flatten_chain
from oracle import exposure_model as ex
from oracle import multiband_model as mb
from random_rigs import random_chain

cv2.ocl.setUseOpenCL(False)


def _check(sizes, corners, masks, images):
    """The bars of the module docstring on one case; returns the gains."""
    N, I, skip = ex.stats(sizes, corners, masks, images)
    want = ex.gains_cv2(sizes, corners, masks, images)
    assert np.array_equal(ex.solve_cv2(N, I, skip), want)
    got = ex.solve(N, I, skip)
    assert np.all(np.abs(got - want) <= 1e-12 * np.abs(want)), (got, want)
    for g, w in zip(got, want):
        assert np.array_equal(ex.lut(g), ex.lut(w)), (g, w)
    assert np.array_equal(got[skip], np.ones(int(skip.sum())))
    return got, (N, I, skip)


def _scene(rng, sizes, corners):
    """One scene seen by every camera at its own brightness scale (0.6-1.4)."""
    W = max(x + w for (w, h), (x, y) in zip(sizes, corners))
    H = max(y + h for (w, h), (x, y) in zip(sizes, corners))
    base = cv2.GaussianBlur(rng.integers(0, 256, (H, W, 3)).astype(np.uint8), (0, 0), 1.5).astype(np.float64)
    return [np.clip(base[y:y + h, x:x + w] * rng.uniform(0.6, 1.4), 0, 255).astype(np.uint8)
            for (w, h), (x, y) in zip(sizes, corners)]


def _masks(rng, sizes):
    """255 with zero and partial (1..254) pixels."""
    out = []
    for w, h in sizes:
        m = np.full((h, w), 255, np.uint8)
        r = rng.random((h, w))
        m[r < float(rng.uniform(0.0, 0.3))] = 0
        m[(r > 0.7) & (r < 0.7 + float(rng.uniform(0.0, 0.2)))] = rng.integers(1, 255)
        out.append(m)
    return out


@pytest.mark.parametrize("seed", range(40))
def test_stats_and_solve_equal_cv2_on_random_rectangles(seed):
    rng = np.random.default_rng(seed)
    n = 2 + seed % 7
    sizes = [(int(rng.integers(10, 90)), int(rng.integers(10, 70))) for _ in range(n)]
    corners = [(int(rng.integers(0, 60)), int(rng.integers(0, 50))) for _ in range(n)]
    _check(sizes, corners, _masks(rng, sizes), _scene(rng, sizes, corners))


def test_contained_disjoint_and_no_common_255_pixel():
    rng = np.random.default_rng(7)
    sizes = [(60, 40), (20, 14), (30, 30), (25, 25)]
    corners = [(0, 0), (10, 8), (100, 0), (115, 10)]   # 1 inside 0; {2, 3} overlap, apart from {0, 1}
    images = _scene(rng, sizes, corners)
    masks = [np.full((h, w), 255, np.uint8) for w, h in sizes]
    gains, (N, I, skip) = _check(sizes, corners, masks, images)
    assert N[0, 2] == N[1, 3] == 0 and N[0, 1] == 20 * 14 and not skip.any()
    # cameras 2 and 3 overlap, but no pixel is 255 in both: N = 1, I = 0, both skipped, gain 1
    masks[2][:, 15:] = 254
    gains, (N, I, skip) = _check(sizes, corners, masks, images)
    assert N[2, 3] == 1 and I[2, 3] == 0 and list(skip) == [False, False, True, True]
    assert gains[2] == gains[3] == 1.0 and gains[0] != 1.0


def test_all_cameras_isolated():
    rng = np.random.default_rng(3)
    sizes = [(20, 20), (20, 20), (20, 20)]
    corners = [(0, 0), (40, 0), (10, 10)]          # 0 and 2 overlap, with masks that never meet at 255
    images = _scene(rng, sizes, corners)
    masks = [np.full((20, 20), 255, np.uint8), np.full((20, 20), 255, np.uint8), np.full((20, 20), 200, np.uint8)]
    gains, (N, I, skip) = _check(sizes, corners, masks, images)
    assert skip.all() and np.array_equal(gains, np.ones(3)) and N[0, 2] == 1


@pytest.mark.parametrize("seed", range(28))
def test_random_rigs_under_every_map_kind(seed):
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    if images[labels[0]].ndim != 3 or images[labels[0]].shape[2] != 3:
        pytest.skip("GainCompensator estimates on 3 channels")
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    frames = [images[l] for l in labels]
    for kind in MAP_KINDS:
        maps = make_maps(images, labels, kind, seed=seed)
        planes = mb.camera_planes(flat.layers, flat.out_w, flat.out_h, frames, [maps.get(l) for l in labels])
        _check(*ex.plane_inputs(planes))


GAINS = [0.0, 0.5, 1.0, 1.5, 2.5, 1 / 3, 0.7, 1.1, 1.2999, 3.0, 255.0, 8e6] + \
    list(np.random.default_rng(0).uniform(0, 3, 40))


@pytest.mark.parametrize("channels", [1, 3, 4])
def test_apply_equals_cv2_on_all_256_values(channels):
    v = np.arange(256, dtype=np.uint8).reshape(16, 16)
    img = v if channels == 1 else np.repeat(v[:, :, None], channels, axis=2)
    for g in GAINS:
        assert np.array_equal(ex.apply(img, g), ex.apply_cv2(img, g)), g
    assert list(ex.lut(0.5)[:6]) == [0, 0, 1, 2, 2, 2]   # halves to even
    assert ex.lut(3.0)[200] == 255 and ex.lut(0.0).max() == 0
    # past v * g = 2^31 cv2's int conversion overflows (to 0 here); the table saturates
    assert np.array_equal(ex.lut(1e9)[1:], np.full(255, 255, np.uint8))


@pytest.mark.parametrize("seams", [None, "voronoi", "graphcut"])
def test_blends_equal_their_cv2_forms(seams):
    st, states, labels, images = chain_case(3, 40, 72, 3)
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    scale = (0.75, 1.0, 1.3)
    frames = [np.clip(images[l] * s, 0, 255).astype(np.uint8) for l, s in zip(labels, scale)]
    maps = [None, make_maps(images, labels, "ramp")[labels[1]], None]
    args = (flat.layers, flat.out_w, flat.out_h, frames, maps)
    gains = ex.camera_gains(flat.layers, flat.out_w, flat.out_h, frames, maps)
    assert gains[0] > 1.0 > gains[2]
    if seams is None:
        got = ex.blend_weighted(*args)
        assert np.array_equal(got, ex.blend_weighted_cv2(*args))
        assert not np.array_equal(got, ex.blend_weighted(*args, gains=[1.0] * 3))
    got = ex.blend_multiband(*args, 3, seams=seams)
    assert np.array_equal(got, ex.blend_multiband_cv2(*args, 3, seams=seams))
    assert not np.array_equal(got, ex.blend_multiband(*args, 3, gains=[1.0] * 3, seams=seams))


# ---- the Python entry points ------------------------------------------------------------------------------
def test_exposure_gains_are_validated():
    st, states, labels, images = chain_case(2, 48, 64, 3)
    assert Stitcher.exposure_gains is None and st._exposure_gains() is None
    st.exposure_gains = {labels[0]: 1.25}
    with pytest.raises(ValueError, match="camera_weights or blend_bands"):
        st._exposure_gains()
    st.blend_bands = 2
    assert st._exposure_gains() == (1.25, 1.0)
    st.blend_bands = 0
    st.camera_weights = {}
    assert st._exposure_gains() == (1.25, 1.0)
    for bad in ({"nope": 1.0}, {labels[0]: -0.5}, {labels[0]: float("nan")}, {labels[0]: float("inf")},
                {labels[0]: True}, {labels[0]: "1"}, [1.0, 1.0]):
        st.exposure_gains = bad
        with pytest.raises(ValueError, match="exposure_gains"):
            st._exposure_gains()
    st.camera_weights = None
    for bad in ({labels[0]: images[labels[0]]}, {l: images[l][:, :-1] for l in labels},
                {l: images[l][:, :, :1] for l in labels}):
        with pytest.raises(ValueError, match="compensate_exposure"):
            st.compensate_exposure(bad)
    with pytest.raises(ValueError, match="camera_weights or blend_bands"):
        st.compensate_exposure(images)
    st.exposure_gains = {labels[0]: 2.0}
    assert st.compensate_exposure(None) is None and st.exposure_gains is None


def test_gains_pickle_and_objects_without_the_attribute_take_the_class_default():
    st, states, labels, images = chain_case(2, 48, 64, 3)
    state = st.__getstate__()
    state.pop("exposure_gains", None)
    clone = Stitcher.__new__(Stitcher)
    clone.__dict__.update(state)
    assert clone._exposure_gains() is None
    st.blend_bands = 3
    st.exposure_gains = {labels[0]: 0.875, labels[1]: 1.0625}
    back = pickle.loads(pickle.dumps(st))
    assert back._exposure_gains() == (0.875, 1.0625)
