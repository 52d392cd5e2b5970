"""Multi-band blend (include/mcs.h mcs_plan_set_multiband), CPU side: the numpy restatement of
oracle/multiband_model.py equals OpenCV's MultiBandBlender bit for bit - pyrDown / pyrUp on int16 on
their own, then the whole blend on synthetic chains, the seeded random rigs, every map kind, 1-6 bands,
1/3/4 channels, clamped band counts, regions feed() shifts and cameras of zero weight; the Python entry
points reject bad requests without a GPU."""
import pickle

import cv2
import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, chain_case, make_maps
from multicamera_stitching_b200 import Stitcher
from multicamera_stitching_b200.plan import flatten_chain
from oracle import multiband_model as mb
from random_rigs import random_chain

cv2.ocl.setUseOpenCL(False)


def _both(st, labels, images, maps, bands):
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    frames, m = [images[l] for l in labels], [maps.get(l) for l in labels]
    return (mb.blend(flat.layers, flat.out_w, flat.out_h, frames, m, bands),
            mb.blend_cv2(flat.layers, flat.out_w, flat.out_h, frames, m, bands))


# ---- pyrDown / pyrUp on int16 ----------------------------------------------------------------------------
@pytest.mark.parametrize("c", [1, 3, 4])
def test_pyramid_steps_equal_cv2_on_every_small_size(c):
    rng = np.random.default_rng(c)
    for h in range(1, 12):
        for w in range(1, 12):
            a = rng.integers(-32768, 32768, size=(h, w) if c == 1 else (h, w, c)).astype(np.int16)
            assert np.array_equal(mb.pyr_down(a), cv2.pyrDown(a)), (h, w)
            assert np.array_equal(mb.pyr_up(a), cv2.pyrUp(a)), (h, w)
            if h > 1 and w > 1:   # the odd destination sizes of the collapse
                ds = (2 * w - 1, 2 * h - 1)
                assert np.array_equal(mb.pyr_up(a, ds), cv2.pyrUp(a, dstsize=ds)), (h, w)


@pytest.mark.parametrize("value", [-32768, -32767, 32766, 32767])
def test_pyramid_steps_saturate_like_cv2(value):
    rng = np.random.default_rng(value & 0xFF)
    for h, w in [(9, 9), (10, 7), (33, 64), (1, 5)]:
        a = np.full((h, w, 3), value, np.int16)
        a[rng.random((h, w)) < 0.2] = -value if value != -32768 else 32767
        assert np.array_equal(mb.pyr_down(a), cv2.pyrDown(a))
        assert np.array_equal(mb.pyr_up(a), cv2.pyrUp(a))


# ---- the blend -------------------------------------------------------------------------------------------
CASES = [  # cameras, height, width, channels, super mode, map kind, bands
    (2, 64, 96, 3, False, "random", 1), (3, 90, 160, 1, False, "binary", 2), (4, 72, 120, 4, False, "ramp", 3),
    (5, 48, 80, 3, False, "absent", 4), (8, 40, 64, 3, False, "mixed", 5), (3, 120, 200, 3, True, "ramp", 6),
    (4, 90, 160, 4, True, "random", 5), (6, 48, 96, 1, True, "mixed", 3), (2, 80, 131, 3, False, "binary", 4),
]


@pytest.mark.parametrize("n,h,w,c,super_mode,kind,bands", CASES)
def test_restatement_equals_cv2_on_synthetic_chains(n, h, w, c, super_mode, kind, bands):
    st, states, labels, images = chain_case(n, h, w, c, super_mode)
    maps = make_maps(images, labels, kind, seed=n * 10 + c)
    got, ref = _both(st, labels, images, maps, bands)
    assert got.shape == ref.shape and np.array_equal(got, ref)


@pytest.mark.parametrize("seed", range(28))
def test_restatement_equals_cv2_on_random_rigs(seed):
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    for i, kind in enumerate(MAP_KINDS):
        bands = 1 + (seed + i) % 6
        maps = make_maps(images, labels, kind, seed=seed)
        got, ref = _both(st, labels, images, maps, bands)
        assert got.shape == ref.shape and np.array_equal(got, ref), (kind, bands)


@pytest.mark.parametrize("bands", range(1, 7))
def test_every_band_count_and_map_kind(bands):
    st, states, labels, images = chain_case(3, 70, 110, 3)
    for kind in MAP_KINDS:
        maps = make_maps(images, labels, kind, seed=bands)
        got, ref = _both(st, labels, images, maps, bands)
        assert np.array_equal(got, ref), kind


def _planes(rng, out_w, out_h, rects, c=3):
    out = []
    for x0, y0, x1, y1 in rects:
        v = rng.integers(0, 256, size=(y1 - y0, x1 - x0, c)).astype(np.uint8)
        w = rng.integers(0, 256, size=(y1 - y0, x1 - x0)).astype(np.int64)
        out.append(((x0, y0, x1, y1), v, w))
    return out


@pytest.mark.parametrize("out_w,out_h,bands", [(1, 1, 5), (2, 1, 5), (3, 2, 4), (5, 7, 6), (8, 3, 8), (17, 9, 8)])
def test_band_count_clamps_on_small_panoramas(out_w, out_h, bands):
    rng = np.random.default_rng(out_w * 100 + out_h)
    n = mb.num_bands(bands, out_w, out_h)
    assert n == min(bands, int(np.ceil(np.log2(max(out_w, out_h)))))
    planes = _planes(rng, out_w, out_h, [(0, 0, out_w, out_h), (out_w // 2, 0, out_w, max(1, out_h // 2))])
    got, det = mb.blend_planes(planes, out_w, out_h, bands, 3)
    assert det["bands"] == n
    assert np.array_equal(got, mb.blend_planes_cv2(planes, out_w, out_h, bands, 3))


@pytest.mark.parametrize("bands", [1, 3, 5])
def test_regions_at_the_right_and_bottom_edges(bands):
    """Rectangles that touch the right and bottom edges of panoramas whose sides are not multiples of 2^n:
    feed()'s region reaches into the padding of the ROI."""
    rng = np.random.default_rng(bands)
    out_w, out_h = 157, 83
    rects = [(0, 0, 100, 60), (90, 20, 157, 83), (140, 70, 157, 83), (3, 80, 40, 83), (156, 0, 157, 83)]
    planes = _planes(rng, out_w, out_h, rects)
    RW, RH = mb.roi_size(mb.num_bands(bands, out_w, out_h), out_w, out_h)
    regions = [mb.feed_region(r, mb.num_bands(bands, out_w, out_h), RW, RH) for r in rects]
    assert any(r[2] > out_w for r in regions) and any(r[3] > out_h for r in regions)
    got, _ = mb.blend_planes(planes, out_w, out_h, bands, 3)
    assert np.array_equal(got, mb.blend_planes_cv2(planes, out_w, out_h, bands, 3))


def test_a_camera_of_zero_weight_everywhere():
    st, states, labels, images = chain_case(3, 90, 160, 3)
    maps = {l: None for l in labels}
    maps[labels[1]] = np.zeros(images[labels[1]].shape[:2], np.uint8)
    got, ref = _both(st, labels, images, maps, 4)
    assert np.array_equal(got, ref)
    # its pixels change nothing: the same rig with that camera black blends the same
    black = dict(images)
    black[labels[1]] = np.zeros_like(images[labels[1]])
    assert np.array_equal(got, _both(st, labels, black, maps, 4)[0])


def test_all_weights_zero_gives_a_black_panorama():
    st, states, labels, images = chain_case(2, 48, 64, 3)
    maps = {l: np.zeros(images[l].shape[:2], np.uint8) for l in labels}
    got, ref = _both(st, labels, images, maps, 3)
    assert np.array_equal(got, ref) and not got.any()


@pytest.mark.parametrize("bands", [2, 5])
def test_the_channel_rule_is_the_per_channel_blend(bands):
    """Channels blend independently under shared weights: each channel of a direct 3-channel blend equals the
    1-channel rule on that channel, and the 4-channel rule's channels 0-2 equal a direct blend of them."""
    rng = np.random.default_rng(bands)
    out_w, out_h = 120, 70
    rects = [(0, 0, 80, 70), (50, 10, 120, 60), (20, 30, 100, 70)]
    planes4 = _planes(rng, out_w, out_h, rects, c=4)
    direct = mb.blend_planes_cv2([(r, v[:, :, :3], w) for r, v, w in planes4], out_w, out_h, bands, 3)
    for ch in range(3):
        one = mb.blend_planes_cv2([(r, v[:, :, ch:ch + 1], w) for r, v, w in planes4], out_w, out_h, bands, 1)
        assert np.array_equal(one[:, :, 0], direct[:, :, ch]), ch
    four = mb.blend_planes_cv2(planes4, out_w, out_h, bands, 4)
    assert np.array_equal(four[:, :, :3], direct)
    last = mb.blend_planes_cv2([(r, v[:, :, 3:4], w) for r, v, w in planes4], out_w, out_h, bands, 1)
    assert np.array_equal(four[:, :, 3], last[:, :, 0])
    assert np.array_equal(mb.blend_planes(planes4, out_w, out_h, bands, 4)[0], four)


def test_the_blender_is_lossy_even_for_one_camera():
    """No reduction to the overwrite: one camera under a full mask comes back changed."""
    rng = np.random.default_rng(7)
    planes = _planes(rng, 96, 64, [(0, 0, 96, 64)])
    planes = [(r, v, np.full_like(w, 255)) for r, v, w in planes]
    got, _ = mb.blend_planes(planes, 96, 64, 3, 3)
    assert np.array_equal(got, mb.blend_planes_cv2(planes, 96, 64, 3, 3))
    assert not np.array_equal(got, planes[0][1])


# ---- the Python entry points ------------------------------------------------------------------------------
def test_blend_bands_is_checked_and_excludes_the_stage_blend():
    st, states, labels, images = chain_case(2, 48, 64, 3)
    assert Stitcher.blend_bands == 0
    st.blend_bands = 3
    assert st._camera_weight_list() == [None, None]   # no maps: 255 everywhere
    st.feather_log2 = 2
    with pytest.raises(ValueError, match="feather_log2"):
        st._camera_weight_list()
    st.feather_log2 = 0
    st.blend_weights = [None]
    with pytest.raises(ValueError, match="blend_weights"):
        st._camera_weight_list()
    st.blend_weights = None
    for bad in (-1, 9, 2.5, True, "3"):
        st.blend_bands = bad
        with pytest.raises(ValueError, match="blend_bands"):
            st._blend_bands()
    st.blend_bands = 0
    assert st._camera_weight_list() is None


def test_objects_without_the_attribute_take_the_class_default():
    st, states, labels, images = chain_case(2, 48, 64, 3)
    state = st.__getstate__()
    state.pop("blend_bands", None)
    clone = Stitcher.__new__(Stitcher)
    clone.__dict__.update(state)
    assert clone._blend_bands() == 0 and clone._camera_weight_list() is None
    assert pickle.loads(pickle.dumps(clone))._blend_bands() == 0
