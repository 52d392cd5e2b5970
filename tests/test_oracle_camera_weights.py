"""Camera-weighted blend (include/mcs.h mcs_plan_set_camera_weights), CPU side: the layer-table model
equals the cv2 chain restatement, reduces to what it should, and the kernel's division is exact;
the Python and C entry points reject bad requests without a GPU."""
import ctypes
import pickle

import cv2
import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, chain_case, layer_model, make_maps
from multicamera_stitching_b200 import Stitcher, _cabi, edge_ramp
from multicamera_stitching_b200.plan import flatten_chain
from oracle import camera_weight_model, stitcher_ref
from random_rigs import random_chain

CASES = [  # cameras, height, width, channels, super mode, map kind
    (2, 64, 96, 3, False, "random"), (3, 90, 160, 1, False, "binary"), (4, 72, 120, 4, False, "ramp"),
    (5, 48, 80, 3, False, "absent"), (8, 40, 64, 3, False, "mixed"), (3, 120, 200, 3, True, "ramp"),
    (4, 90, 160, 4, True, "random"), (6, 48, 96, 1, True, "mixed"), (2, 80, 131, 3, False, "binary"),
]


@pytest.mark.parametrize("n,h,w,c,super_mode,kind", CASES)
def test_layer_model_equals_the_cv2_chain(n, h, w, c, super_mode, kind):
    st, states, labels, images = chain_case(n, h, w, c, super_mode)
    maps = make_maps(images, labels, kind, seed=n * 10 + c)
    got, contrib, most = layer_model(st, labels, images, maps)
    ref = camera_weight_model.chain(states, labels, images, maps)
    assert got.shape == ref.shape == stitcher_ref.stitch_chain(states, labels, images).shape
    assert np.array_equal(got, ref)
    assert sum(contrib) > 0 and most >= 1


@pytest.mark.parametrize("seed", range(28))
def test_layer_model_equals_the_cv2_chain_on_random_rigs(seed):
    """The seeded random rigs of the overwrite fuzz (rotations, anisotropic scales, perspective, mirrored cameras,
    odd widths, 1/3/4 channels), super-mode crops trimmed so that they keep several cameras, under every map kind.
    ``most`` is held against a per-pixel count of the cv2 chain's planes."""
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    for kind in MAP_KINDS:
        maps = make_maps(images, labels, kind, seed=seed)
        got, contrib, most = layer_model(st, labels, images, maps)
        planes = camera_weight_model.chain_planes(states, labels, images, maps)
        ref = camera_weight_model.chain(states, labels, images, maps)
        assert got.shape == ref.shape and np.array_equal(got, ref), kind
        count = sum((r & (w > 0)).astype(np.int64) for _, w, r in planes)
        assert most == int(count.max()) and sum(contrib) == int(count.sum()), kind
        assert 1 <= most <= camera_weight_model.MAX_CONTRIBUTORS, kind


@pytest.mark.parametrize("j", [0, 1, 2])
def test_one_camera_with_weight_gives_its_warp_inside_its_rectangle(j):
    st, states, labels, images = chain_case(3, 90, 160, 3)
    maps = {l: (None if i == j else np.zeros(images[l].shape[:2], np.uint8)) for i, l in enumerate(labels)}
    got, contrib, most = layer_model(st, labels, images, maps)
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    l = flat.layers[j]
    x0, y0, x1, y1 = l.rect
    want = np.zeros_like(got)
    if j == 0:
        want[y0:y1, x0:x1] = images[labels[0]][y0 - l.oy:y1 - l.oy, x0 - l.ox:x1 - l.ox]
    else:
        warped = cv2.warpPerspective(images[labels[j]], states[j - 1]["cachedAH"], tuple(states[j - 1]["ABSize"]))
        want[y0:y1, x0:x1] = warped[y0 - l.oy:y1 - l.oy, x0 - l.ox:x1 - l.ox]
    assert np.array_equal(got, want)
    assert most == 1 and all(v == 0 for k, v in enumerate(contrib) if k != j)


def test_zero_map_equals_the_overwrite_with_a_black_camera():
    st, states, labels, images = chain_case(2, 90, 160, 3)
    maps = {labels[0]: None, labels[1]: np.zeros(images[labels[1]].shape[:2], np.uint8)}
    got, _, _ = layer_model(st, labels, images, maps)
    black = dict(images)
    black[labels[1]] = np.zeros_like(images[labels[1]])
    assert np.array_equal(got, stitcher_ref.stitch_chain(states, labels, black))


def test_one_contributor_is_exact_and_equal_weights_round_half_up():
    st, states, labels, images = chain_case(3, 90, 160, 3)
    maps = make_maps(images, labels, "random", seed=5)
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    planes = [camera_weight_model.layer_planes(l, images[labels[l.cam]], maps[labels[l.cam]], flat.out_w, flat.out_h)
              for l in flat.layers]
    V = np.zeros((len(planes), flat.out_h, flat.out_w, 3), np.int64)
    Wt = np.zeros((len(planes), flat.out_h, flat.out_w), np.int64)
    for k, ((x0, y0, x1, y1), v, w) in enumerate(planes):
        V[k, y0:y1, x0:x1], Wt[k, y0:y1, x0:x1] = v, w
    got, _, _ = layer_model(st, labels, images, maps)
    n = (Wt > 0).sum(axis=0)
    one = n == 1
    assert one.sum() > 1000
    k1 = np.argmax(Wt > 0, axis=0)
    single = np.take_along_axis(V, k1[None, ..., None], axis=0)[0]
    assert np.array_equal(got[one], single[one])
    # two cameras of equal weight: (v0 + v1 + 1) // 2
    maps = {l: None for l in labels}
    got, _, _ = layer_model(st, labels, images, maps)
    planes = [camera_weight_model.layer_planes(l, images[labels[l.cam]], None, flat.out_w, flat.out_h)
              for l in flat.layers]
    V[:], Wt[:] = 0, 0
    for k, ((x0, y0, x1, y1), v, w) in enumerate(planes):
        V[k, y0:y1, x0:x1], Wt[k, y0:y1, x0:x1] = v, w
    pair = ((Wt == 255).sum(axis=0) == 2) & ((Wt > 0).sum(axis=0) == 2)
    assert pair.sum() > 1000
    a, b = [np.take_along_axis(V, idx[None, ..., None], axis=0)[0]
            for idx in (np.argmax(Wt > 0, axis=0), Wt.shape[0] - 1 - np.argmax((Wt > 0)[::-1], axis=0))]
    assert np.array_equal(got[pair], ((a + b + 1) // 2)[pair])


def test_mulhi_division_is_exact_over_every_reachable_numerator():
    top = camera_weight_model.MAX_CONTRIBUTORS * 255
    for S in range(2, top + 1):
        n = np.arange(255 * S + S // 2 + 1, dtype=np.uint64)
        assert np.array_equal(camera_weight_model.mulhi_div(n, S), n // np.uint64(S)), S


def test_edge_ramp():
    m = edge_ramp((5, 7), 2)
    assert m.dtype == np.uint8 and m.shape == (5, 7)
    assert m[0, 0] == 127 and m[1, 1] == 255 and m[2, 0] == 127 and m[2, 3] == 255
    assert np.array_equal(edge_ramp((3, 3, 3), 1), np.full((3, 3), 255, np.uint8))
    with pytest.raises(ValueError):
        edge_ramp((4, 4), 0)


def test_camera_weights_are_checked_and_pickled():
    st, states, labels, images = chain_case(3, 60, 96, 3)
    assert Stitcher.camera_weights is None and st._camera_weight_list() is None
    good = {labels[1]: edge_ramp(images[labels[1]].shape, 8)}
    st.camera_weights = good
    lst = st._camera_weight_list()
    assert lst[0] is None and lst[2] is None and lst[1] is good[labels[1]]
    for bad in ({labels[1]: np.zeros((5, 5), np.uint8)}, {"nope": None},
                {labels[0]: np.zeros(images[labels[0]].shape[:2], np.float32)}):
        st.camera_weights = bad
        with pytest.raises(ValueError):
            st._camera_weight_list()
    st.camera_weights = good
    st.feather_log2 = 2
    with pytest.raises(ValueError):
        st._camera_weight_list()
    st.feather_log2 = 0
    st.blend_weights = [None, None]
    with pytest.raises(ValueError):
        st._camera_weight_list()
    st.blend_weights = None
    back = pickle.loads(pickle.dumps(st))
    assert np.array_equal(back.camera_weights[labels[1]], good[labels[1]])


def test_set_camera_weights_rejects_a_null_plan_without_a_gpu():
    lib = _cabi.load()
    assert lib.mcs_plan_set_camera_weights(None, None, None) == -1
    assert "plan is NULL" in lib.mcs_last_error().decode()
    maps = (ctypes.c_void_p * 1)()
    assert lib.mcs_plan_set_camera_weights(None, maps, None) == -1

