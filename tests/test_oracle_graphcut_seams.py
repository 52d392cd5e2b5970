"""Graph-cut seam masks (include/mcs.h mcs_plan_set_graphcut_seams), CPU side: the integer restatement
``oracle/graphcut_seam_model.find_graphcut`` equals OpenCV's GraphCutSeamFinder("COST_COLOR") on every pixel on textured
content (random 2-6-camera rectangle sets, masks with holes and zero borders, the seeded random rigs); on flat and
identical content, where several cuts cost the minimum, cv2's cut still costs the minimum and the restatement's is
the minimal source side; the restatement does not depend on the max-flow algorithm; the Python entry points reject
bad requests without a GPU."""
import pickle

import cv2
import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, chain_case, make_maps
from multicamera_stitching_b200 import Stitcher
from multicamera_stitching_b200.plan import flatten_chain
from oracle import multiband_model as mb
from oracle import graphcut_seam_model, seam_model
from random_rigs import random_chain

cv2.ocl.setUseOpenCL(False)


def _textured(rng, sizes, corners, noise=24):
    """Every camera's view of one blurred scene plus its own noise: content on which the cameras nearly agree."""
    W = max(x + w for (w, h), (x, y) in zip(sizes, corners))
    H = max(y + h for (w, h), (x, y) in zip(sizes, corners))
    base = cv2.GaussianBlur(rng.integers(0, 256, (H, W, 3)).astype(np.uint8), (0, 0), 2)
    return [np.clip(base[y:y + h, x:x + w].astype(int) + rng.integers(-noise, noise + 1, (h, w, 3)), 0, 255)
            .astype(np.uint8) for (w, h), (x, y) in zip(sizes, corners)]


def _masks(rng, sizes, holes):
    out = []
    for w, h in sizes:
        m = rng.integers(1, 256, (h, w)).astype(np.uint8)
        if holes:
            m[rng.random((h, w)) < 0.05] = 0
            m[:, :2] = 0
            m[-1, :] = 0
            y, x = int(rng.integers(0, h)), int(rng.integers(0, w))
            m[y:y + h // 4, x:x + w // 4] = 0
        out.append(m)
    return out


def _check(sizes, corners, masks, images):
    got, pairs = graphcut_seam_model.find_graphcut(sizes, corners, masks, images, details=True)
    ref = graphcut_seam_model.find_graphcut_cv2(sizes, corners, masks, images)
    assert all(np.array_equal(g, r) for g, r in zip(got, ref)), [int((g != r).sum()) for g, r in zip(got, ref)]
    for g, m in zip(got, masks):   # the finder only zeroes
        assert np.all((g == 0) | (g == m))
    return got, pairs


@pytest.mark.parametrize("seed", range(24))
def test_restatement_equals_cv2_on_random_rectangles(seed):
    rng = np.random.default_rng(seed)
    n = 2 + seed % 5
    sizes = [(int(rng.integers(12, 80)), int(rng.integers(12, 70))) for _ in range(n)]
    corners = [(int(rng.integers(0, 60)), int(rng.integers(0, 50))) for _ in range(n)]
    images = _textured(rng, sizes, corners)
    got, pairs = _check(sizes, corners, _masks(rng, sizes, holes=seed % 2 == 1), images)
    assert pairs or n == 2


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
    if images[labels[0]].ndim != 3 or images[labels[0]].shape[2] != 3:
        pytest.skip("the colour cost takes 3 channels")
    planes = _rig_planes(st, labels, images, make_maps(images, labels, MAP_KINDS[seed % 7], seed=seed))
    _check(*graphcut_seam_model.plane_inputs(planes))


def _pair(rng, kind, w=46, h=30, shift=(18, 3)):
    sizes = [(w, h), (w, h)]
    corners = [(0, 0), shift]
    if kind == "flat":
        images = [np.full((h, w, 3), 77, np.uint8)] * 2
    else:   # identical: the same frame in both cameras, so the overlap differs wherever the shift moves content
        f = rng.integers(0, 256, (h, w, 3)).astype(np.uint8)
        f[:, ::2] = f[:, :1]
        images = [f, f]
    masks = [np.full((h, w), 255, np.uint8), np.full((h, w), 255, np.uint8)]
    if rng.random() < 0.5:
        masks[0][rng.random((h, w)) < 0.03] = 0
    return sizes, corners, masks, images


@pytest.mark.parametrize("seed", range(24))
def test_flat_and_identical_content_cv2_cuts_and_the_minimal_side(seed):
    """Pin cv2's observable labels with terminal edges of 2^30 (every real capacity is below 2^21) and solve again.
    With full masks the value is unchanged: cv2's cut is a minimum cut, only another one than the minimal source
    side.  With zero holes in a mask it can cost a few units more (here seed 12, by 2; over the first 48 seeds of
    this generator 4 of the 8 flat pairs with holes, by 2-6): cv2's search leaves some pixels that are in neither of its trees on the costlier side.  Every pixel cv2
    puts on the sink side is outside the restatement's S, and S is a minimum cut."""
    rng = np.random.default_rng(100 + seed)
    sizes, corners, masks, images = _pair(rng, ("flat", "identical")[seed % 2])
    roi = seam_model.overlap(sizes[0], corners[0], sizes[1], corners[1])
    s1, s2 = graphcut_seam_model.sub(masks[0], corners[0], roi), graphcut_seam_model.sub(masks[1], corners[1], roi)
    i1, i2 = graphcut_seam_model.sub(images[0], corners[0], roi), graphcut_seam_model.sub(images[1], corners[1], roi)
    M, source, sink, n = graphcut_seam_model.graphcut_graph(s1, s2, i1, i2)
    value, reach = graphcut_seam_model.min_cut(M, source, sink)
    S = reach[:n].reshape(s1.shape)
    o1, o2 = graphcut_seam_model.find_graphcut_cv2(sizes, corners, masks, images)
    g = graphcut_seam_model.GAP
    c1, c2 = graphcut_seam_model.sub(o1, corners[0], roi), graphcut_seam_model.sub(o2, corners[1], roi)
    inner = np.zeros(s1.shape, bool)
    inner[g:-g, g:-g] = True
    both = inner & (s1 != 0) & (s2 != 0)
    cv_source = both & (c2 == 0)    # cv2 zeroed camera j: the pixel is on its source side
    cv_sink = both & (c1 == 0)
    assert not (cv_source & cv_sink).any() and np.array_equal(cv_source | cv_sink, both)
    Mp, _, _, _ = graphcut_seam_model.graphcut_graph(s1, s2, i1, i2, pin_source=cv_source, pin_sink=cv_sink)
    pinned = graphcut_seam_model.min_cut(Mp, source, sink)[0]
    if masks[0].all():
        assert pinned == value
    else:
        assert value <= pinned < value + graphcut_seam_model.PENALTY
    assert not (S & cv_sink).any()
    Mo, _, _, _ = graphcut_seam_model.graphcut_graph(s1, s2, i1, i2, pin_source=S, pin_sink=~S)
    assert graphcut_seam_model.min_cut(Mo, source, sink)[0] == value


@pytest.mark.parametrize("seed", range(6))
def test_the_cut_does_not_depend_on_the_flow_algorithm(seed):
    rng = np.random.default_rng(200 + seed)
    if seed % 2:
        sizes, corners, masks, images = _pair(rng, ("flat", "identical")[seed % 3 == 0])
    else:
        sizes = [(40, 36), (44, 30), (30, 40)]
        corners = [(0, 0), (20, 6), (8, 14)]
        images = _textured(rng, sizes, corners)
        masks = _masks(rng, sizes, holes=True)
    a = graphcut_seam_model.find_graphcut(sizes, corners, masks, images, method="dinic")
    b = graphcut_seam_model.find_graphcut(sizes, corners, masks, images, method="edmonds_karp")
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_blend_with_graphcut_seams_equals_cv2():
    st, states, labels, images = chain_case(3, 40, 72, 3)
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    frames = [images[l] for l in labels]
    maps = [None] * len(labels)
    got = graphcut_seam_model.blend_graphcut(flat.layers, flat.out_w, flat.out_h, frames, maps, 3)
    assert np.array_equal(got, graphcut_seam_model.blend_graphcut_cv2(flat.layers, flat.out_w, flat.out_h, frames, maps, 3))
    assert not np.array_equal(got, seam_model.blend(flat.layers, flat.out_w, flat.out_h, frames, maps, 3))


# ---- the Python entry points ------------------------------------------------------------------------------
def test_find_graphcut_seams_validates_its_frames_and_mode():
    st, states, labels, images = chain_case(2, 48, 64, 3)
    assert Stitcher.graphcut_seams is None and st._graphcut_seams() is None
    st.find_graphcut_seams(images)
    with pytest.raises(ValueError, match="blend_bands"):
        st._graphcut_seams()
    st.blend_bands = 3
    digest, frames = st._graphcut_seams()
    assert len(frames) == 2 and all(not f.flags.writeable for f in frames)
    assert all(np.array_equal(f, images[l]) for f, l in zip(frames, labels))
    st.voronoi_seams = True
    with pytest.raises(ValueError, match="voronoi_seams"):
        st._graphcut_seams()
    st.voronoi_seams = False
    # the digest follows the content and is computed once
    images[labels[0]][0, 0, 0] ^= 1
    assert st._graphcut_seams()[0] == digest
    st.find_graphcut_seams(images)
    assert st._graphcut_seams()[0] != digest
    for bad in ({labels[0]: images[labels[0]]},
                {l: images[l][:, :-1] for l in labels},
                {l: images[l][:, :, :1] for l in labels},
                {l: images[l].astype(np.int16) for l in labels}):
        with pytest.raises(ValueError, match="find_graphcut_seams"):
            st.find_graphcut_seams(bad)
    st.find_graphcut_seams(None)
    assert st._graphcut_seams() is None


def test_objects_without_the_attribute_take_the_class_default():
    st, states, labels, images = chain_case(2, 48, 64, 3)
    state = st.__getstate__()
    state.pop("graphcut_seams", None)
    clone = Stitcher.__new__(Stitcher)
    clone.__dict__.update(state)
    assert clone._graphcut_seams() is None
    assert pickle.loads(pickle.dumps(clone))._graphcut_seams() is None
    st.blend_bands = 2
    st.find_graphcut_seams(images)
    back = pickle.loads(pickle.dumps(st))
    assert back._graphcut_seams()[0] == st._graphcut_seams()[0]
