"""Voronoi seam masks (include/mcs.h mcs_plan_set_voronoi_seams), CPU side: the numpy restatement
``oracle/seam_model.find`` equals OpenCV's VoronoiSeamFinder bit for bit on random rectangles and masks
(2-8 cameras, contained and disjoint rectangles, empty, full, non-binary and checkerboard masks, ROIs at the
panorama edges, exact ties) and on the seeded random rigs under every map kind; its output keeps no pixel in two
masks and leaves surviving weights as they were; the multi-band blend of the cut weights equals cv2's; the
Python entry points reject bad requests without a GPU."""
import pickle

import cv2
import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, chain_case, make_maps
from multicamera_stitching_b200 import Stitcher
from multicamera_stitching_b200.plan import flatten_chain
from oracle import multiband_model as mb
from oracle import seam_model
from random_rigs import random_chain

cv2.ocl.setUseOpenCL(False)


def _check(sizes, corners, masks):
    got, pairs = seam_model.find(sizes, corners, masks, details=True)
    ref = seam_model.find_cv2(sizes, corners, masks)
    assert all(np.array_equal(g, r) for g, r in zip(got, ref)), [int((g != r).sum()) for g, r in zip(got, ref)]
    # properties: no pixel non-zero in two masks, every survivor its input weight
    H = max(c[1] + s[1] for s, c in zip(sizes, corners))
    W = max(c[0] + s[0] for s, c in zip(sizes, corners))
    count = np.zeros((H, W), np.int64)
    for g, m, (w, h), (x, y) in zip(got, masks, sizes, corners):
        assert np.all((g == 0) | (g == m))
        count[y:y + h, x:x + w] += g != 0
    assert count.max() <= 1
    return got, pairs


def _mask(rng, kind, h, w):
    if kind == "full":
        return np.full((h, w), 255, np.uint8)
    if kind == "empty":
        return np.zeros((h, w), np.uint8)
    if kind == "values":
        m = rng.integers(0, 256, size=(h, w)).astype(np.uint8)
        m[rng.random((h, w)) < 0.3] = 0
        return m
    if kind == "checker":
        yy, xx = np.mgrid[0:h, 0:w]
        return (((yy // (1 + h % 3) + xx // (1 + w % 4)) % 2) * 7).astype(np.uint8)
    m = np.zeros((h, w), np.uint8)   # "partial": a block of 7
    m[h // 3:, :w // 2] = 7
    return m


MASK_KINDS = ("full", "empty", "values", "checker", "partial")


@pytest.mark.parametrize("seed", range(40))
def test_restatement_equals_cv2_on_random_rectangles(seed):
    rng = np.random.default_rng(seed)
    n = 2 + seed % 7
    sizes = [(int(rng.integers(3, 90)), int(rng.integers(3, 70))) for _ in range(n)]
    corners = [(int(rng.integers(0, 70)), int(rng.integers(0, 50))) for _ in range(n)]
    masks = [_mask(rng, MASK_KINDS[int(rng.integers(0, 5))], h, w) for w, h in sizes]
    cv2.ipp.setUseIPP(bool(seed % 2))
    try:
        _check(sizes, corners, masks)
    finally:
        cv2.ipp.setUseIPP(True)


def test_contained_disjoint_and_edge_rectangles():
    rng = np.random.default_rng(5)
    # a rectangle inside another, one disjoint from both, ROIs at the panorama's left / top edge
    sizes = [(100, 80), (30, 20), (40, 40), (25, 90), (100, 12)]
    corners = [(0, 0), (35, 30), (150, 10), (0, 0), (0, 68)]
    for kinds in [("full",) * 5, ("values", "full", "checker", "partial", "values"), ("empty", "full", "full", "values", "checker")]:
        masks = [_mask(rng, k, h, w) for k, (w, h) in zip(kinds, sizes)]
        got, pairs = _check(sizes, corners, masks)
        assert [(i, j) for i, j, _ in pairs] == [(0, 1), (0, 3), (0, 4), (3, 4)]
    # the contained camera keeps nothing under full masks: the outer one is nearer everywhere it is unique
    full = [np.full((h, w), 255, np.uint8) for w, h in sizes[:2]]
    got, _ = _check(sizes[:2], corners[:2], full)
    assert not got[1].any() and got[0].all()


@pytest.mark.parametrize("w", [4, 7, 20])
def test_exact_ties_go_to_the_later_camera(w):
    """Two cameras side by side whose overlap is exactly halfway between their unique parts."""
    sizes = [(20 + w, 10), (20 + w, 10)]
    corners = [(0, 0), (20, 0)]
    masks = [np.full((10, 20 + w), 255, np.uint8), np.full((10, 20 + w), 255, np.uint8)]
    got, _ = _check(sizes, corners, masks)
    if w % 2 == 1:   # the middle column is a tie: it is cut from camera 0
        mid = 20 + w // 2
        assert not got[0][:, mid].any() and got[1][:, mid - 20].all()


def test_both_unique_parts_empty_everywhere_ties():
    """Identical rectangles with full masks: both u are empty, the distances tie and camera 0 loses all."""
    sizes = [(30, 20)] * 3
    corners = [(5, 5)] * 3
    masks = [np.full((20, 30), v, np.uint8) for v in (9, 200, 255)]
    got, _ = _check(sizes, corners, masks)
    assert not got[0].any() and not got[1].any() and np.array_equal(got[2], masks[2])


@pytest.mark.parametrize("col,kept", [(10, [10, 20, 21, 22, 23, 24]), (9, [9])])
def test_the_submask_reaches_ten_pixels_beyond_the_overlap(col, kept):
    """Camera 0's only unique pixels are one column ``20 - col`` pixels left of the overlap: at 10 they are inside the
    submask and win the left quarter of the overlap; at 11 the submask misses them and camera 0 loses it all."""
    sizes, corners = [(40, 20), (40, 20)], [(0, 0), (20, 0)]
    m0 = np.zeros((20, 40), np.uint8)
    m0[:, col] = 255
    m0[:, 20:] = 200
    got, _ = _check(sizes, corners, [m0, np.full((20, 40), 255, np.uint8)])
    assert list(np.nonzero(got[0][0])[0]) == kept


def test_the_bound_is_refused():
    sizes = [(32740, 4), (32740, 4)]
    corners = [(0, 0), (0, 0)]
    assert not seam_model.supported(sizes, corners)
    with pytest.raises(ValueError, match="32768"):
        seam_model.find(sizes, corners, [np.ones((4, 32740), np.uint8)] * 2)
    assert seam_model.supported([(32726, 1), (32726, 1)], corners)


def _rig_planes(st, labels, images, maps):
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    return mb.camera_planes(flat.layers, flat.out_w, flat.out_h, [images[l] for l in labels],
                            [maps.get(l) for l in labels])


@pytest.mark.parametrize("seed", range(28))
def test_restatement_equals_cv2_on_random_rigs(seed):
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    for kind in MAP_KINDS:
        planes = _rig_planes(st, labels, images, make_maps(images, labels, kind, seed=seed))
        _check(*seam_model.plane_inputs(planes))


@pytest.mark.parametrize("seed", range(28))
def test_blend_with_seams_equals_cv2_on_random_rigs(seed):
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    frames = [images[l] for l in labels]
    kind = MAP_KINDS[seed % len(MAP_KINDS)]
    m = make_maps(images, labels, kind, seed=seed)
    maps = [m.get(l) for l in labels]
    bands = 1 + seed % 6
    got = seam_model.blend(flat.layers, flat.out_w, flat.out_h, frames, maps, bands)
    ref = seam_model.blend_cv2(flat.layers, flat.out_w, flat.out_h, frames, maps, bands)
    assert got.shape == ref.shape and np.array_equal(got, ref), (kind, bands)


@pytest.mark.parametrize("c,bands", [(1, 2), (3, 4), (4, 6), (3, 1)])
def test_blend_with_seams_on_chains_and_channels(c, bands):
    st, states, labels, images = chain_case(4, 72, 120, c)
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    frames = [images[l] for l in labels]
    maps = [None] * len(labels)
    got = seam_model.blend(flat.layers, flat.out_w, flat.out_h, frames, maps, bands)
    assert np.array_equal(got, seam_model.blend_cv2(flat.layers, flat.out_w, flat.out_h, frames, maps, bands))
    # the seams change the panorama: the overlaps are no longer averaged at level 0
    assert not np.array_equal(got, mb.blend(flat.layers, flat.out_w, flat.out_h, frames, maps, bands))


# ---- the Python entry points ------------------------------------------------------------------------------
def test_voronoi_seams_needs_the_multiband_blend():
    st, states, labels, images = chain_case(2, 48, 64, 3)
    assert Stitcher.voronoi_seams is False
    assert st._voronoi_seams() is False
    st.voronoi_seams = True
    with pytest.raises(ValueError, match="blend_bands"):
        st._voronoi_seams()
    st.blend_bands = 3
    assert st._voronoi_seams() is True
    for bad in (1, "yes", None, 2.0):
        st.voronoi_seams = bad
        with pytest.raises(ValueError, match="voronoi_seams"):
            st._voronoi_seams()


def test_objects_without_the_attribute_take_the_class_default():
    st, states, labels, images = chain_case(2, 48, 64, 3)
    state = st.__getstate__()
    state.pop("voronoi_seams", None)
    clone = Stitcher.__new__(Stitcher)
    clone.__dict__.update(state)
    assert clone._voronoi_seams() is False
    assert pickle.loads(pickle.dumps(clone))._voronoi_seams() is False
