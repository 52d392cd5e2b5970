"""GPU: seeded random chains against the reference's cv2 chain (oracle/stitcher_ref.py).  Random
camera counts, frame sizes, channel counts, canvas offsets, super mode and homographies well outside
the benchmark's near-identity ones (rotation, anisotropic scale, perspective, mirrored axes), each
through the automatic variant and, where the plan allows it, with the tiled and the gather kernels
forced.  Everything must be bit-exact."""
import numpy as np
import pytest

from helpers import compare_u8
from multicamera_stitching_b200 import _cabi
from oracle import stitcher_ref
from random_rigs import random_chain

pytestmark = pytest.mark.gpu

TILED_SEEDS = []   # seeds whose chain also ran through the forced tiled variant


@pytest.mark.parametrize("seed", range(28))
def test_random_chain_matches_cv2(cuda_device, seed):
    made = random_chain(seed)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    try:
        ref = stitcher_ref.stitch_chain(states, labels, images)
    except (ValueError, cv2_error()) as e:      # the reference itself fails on this geometry
        with pytest.raises(Exception):
            st.stitch(images)
        pytest.skip("reference raises here too: %s" % (e,))
    got = st.stitch(images)
    assert compare_u8(got, ref) == (0, 1.0)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    variants = [1] + ([2] if plan.handle.tiled_status() == "" else [])
    ran = []
    for v in variants:
        plan.handle.force_variant(v)
        try:
            out = st.stitch(images)
        except _cabi.McsError as e:              # the buffers of this call rule the tiled variant out
            assert v == 2 and "unavailable" in str(e)   # (row pitch not a multiple of 16 bytes)
            continue
        assert compare_u8(out, ref) == (0, 1.0), "variant %d" % v
        assert plan.handle.last_variant() == v
        ran.append(v)
    plan.handle.force_variant(0)
    assert 1 in ran
    if 2 in ran:
        TILED_SEEDS.append(seed)


def test_fuzz_exercised_the_tiled_variant(cuda_device):
    assert len(TILED_SEEDS) >= 10, TILED_SEEDS


def cv2_error():
    import cv2
    return cv2.error


@pytest.mark.parametrize("seed", range(20))
def test_random_chain_blend_modes_match_the_specification(cuda_device, seed):
    """The blend modes on the same random chains (rotations, anisotropic scales, perspective, mirrored cameras, super
    mode): the distance ramp through whichever form the plan takes - BAND tiles of the tiled kernel, or the
    overwrite pass + band pass where the plan cannot be fused (more than two outer cameras per tile, odd rows) - and,
    where the fused form applies, random per-stage weight maps."""
    from oracle import feather_model
    made = random_chain(seed)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    log2 = 1 + seed % 4
    try:
        ref = feather_model.feather_chain(states, labels, images, log2)
    except (ValueError, cv2_error()) as e:
        pytest.skip("the specification's cv2 chain raises on this geometry: %s" % (e,))
    st.feather_log2 = log2
    try:
        got = st.stitch(images)
    except _cabi.McsError as e:
        # cut (super-mode) rectangles exist in the fused form only: a plan that cannot take it says so
        assert "fused band form" in str(e)
        pytest.skip(str(e))
    assert compare_u8(got, ref) == (0, 1.0)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    if plan.handle.tiled_stats()["band_fused"]:
        rng = np.random.default_rng(seed)
        F = 1 << log2
        maps, shapeB = [], images[labels[0]].shape[:2]
        for sb in st.stitchers:
            m = rng.integers(0, F + 1, size=shapeB).astype(np.uint8)
            m[rng.random(shapeB) < 0.6] = F
            maps.append(m)
            shapeB = sb.result_shape()[:2]
        st.blend_weights = maps
        try:
            got = st.stitch(images)
        except _cabi.McsError as e:
            assert "fused band form" in str(e)      # dense maps can need more than two outer cameras per tile
            return
        assert compare_u8(got, feather_model.feather_chain(states, labels, images, log2, maps)) == (0, 1.0)
