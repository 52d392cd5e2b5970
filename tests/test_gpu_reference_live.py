"""The CUDA path against the REFERENCE'S OWN ``Stitcher`` class, run live on the GPU box.

``oracle/_ref`` (the reference's ``StitcherClass.py`` made importable by ``oracle/build_ref.py``, with the stand-in
logging module and a byte copy of the reference's ``Utils.py``) is a build output that travels with the repository
snapshot; the reference tree itself does not.  Where that output is present, the reference class is calibrated by
its own ``calibrate_stitcher`` with the stage homographies of the synthetic rigs and its ``stitch(images_dic)`` is
held against the product's, bit for bit.  Where it is absent (a clean checkout: the repository does not ship the
reference) these tests skip; what remains checked against the reference there is the committed fixture
tests/golden/chain_ref.npz (tests/test_golden.py), the panoramas of three chains, not the cases below."""
import numpy as np
import pytest

from multicamera_stitching_b200 import synthetic
from oracle import build_ref

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    mod = build_ref.load()
    if mod is None:
        pytest.skip("oracle/_ref was not built (python oracle/build_ref.py where the reference tree is present)")
    return mod


@pytest.mark.parametrize("n,h,w,super_mode,kind", [
    (3, 720, 1280, False, "smooth"),     # BASELINE config 1
    (3, 720, 1280, False, "noise"),
    (6, 270, 480, False, "noise"),
    (4, 180, 320, True, "noise"),        # super mode: the reference returns the cropped view
    (8, 135, 240, False, "smooth"),
])
def test_cuda_chain_equals_the_reference_class(cuda_device, ref, n, h, w, super_mode, kind):
    st, homographies, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, super_mode=super_mode, kind=kind)
    rs = build_ref.calibrated_stitcher(ref, images, homographies, super_mode=super_mode)
    for frame_index in (0, 1):
        frames = synthetic.make_frames(n, h, w, 3, frame_index=frame_index, kind=kind)
        want = rs.stitch(frames)
        got = st.stitch(frames)
        assert got.shape == want.shape and got.dtype == want.dtype
        assert np.array_equal(got, want)


def test_cuda_pair_equals_the_reference_class(cuda_device, ref):
    st, homographies, labels, images = synthetic.synthetic_stitcher(2, 200, 300, 3, kind="noise")
    rs = build_ref.calibrated_stitcher(ref, images, homographies)
    pair = (images[labels[0]], images[labels[1]])
    assert np.array_equal(st.stitchers[0].stitch(pair), rs.stitchers[0].stitch(images=pair))


def test_cuda_match_keypoints_equals_the_reference_class(cuda_device, ref):
    """``StitcherBase.matchKeypoints`` (StitcherClass.py:405-448) with float descriptors, the reference's own SIFT
    branch: the match list of the GPU path (L2 2-NN + ratio test) equals the reference method's; the homography
    agrees with the reference's ``findHomography`` result within 0.5 px on the matched points' extent (different
    RANSAC sampling, same inliers' least-squares fit)."""
    from multicamera_stitching_b200 import StitcherBase
    rng = np.random.default_rng(5)
    nA, nB = 700, 800
    featB = np.rint(rng.normal(0, 40, (nB, 128)).clip(0, 255)).astype(np.float32)      # SIFT descriptors are
    perm = rng.permutation(nB)[:nA]                                                    # integer-valued floats
    featA = np.rint((featB[perm] + rng.normal(0, 6, (nA, 128))).clip(0, 255)).astype(np.float32)
    featA[600:] = np.rint(rng.normal(0, 40, (100, 128)).clip(0, 255)).astype(np.float32)
    H_true = np.array([[0.97, 0.02, 31.0], [-0.015, 1.01, 7.5], [1e-5, -2e-5, 1.0]])
    kpsA = rng.uniform(0, 600, (nA, 2)).astype(np.float32)
    proj = np.c_[kpsA, np.ones(nA)] @ H_true.T
    kpsB = np.zeros((nB, 2), np.float32)
    kpsB[perm] = (proj[:, :2] / proj[:, 2:]).astype(np.float32) + rng.normal(0, 0.3, (nA, 2)).astype(np.float32)
    H0, m0, s0 = ref.StitcherBase().matchKeypoints(kpsA=kpsA, kpsB=kpsB, featuresA=featA, featuresB=featB,
                                                   ratio=0.75, reprojThresh=3.0)
    H1, m1, s1 = StitcherBase().matchKeypoints(kpsA=kpsA, kpsB=kpsB, featuresA=featA, featuresB=featB,
                                               ratio=0.75, reprojThresh=3.0)
    assert [tuple(m) for m in m1] == [tuple(m) for m in m0] and len(m0) > 400
    corners = np.array([[0, 0, 1], [600, 0, 1], [600, 600, 1], [0, 600, 1]], dtype=np.float64)
    p0, p1 = corners @ np.asarray(H0).T, corners @ np.asarray(H1).T
    assert np.abs(p0[:, :2] / p0[:, 2:] - p1[:, :2] / p1[:, 2:]).max() < 0.5
    assert np.asarray(s1).shape == np.asarray(s0).shape
    assert (np.asarray(s1).ravel() != np.asarray(s0).ravel()).mean() < 0.02      # inlier masks agree on >= 98 %


@pytest.mark.parametrize("n,super_mode", [(3, False), (4, True)])
def test_cuda_debug_overlays_equal_the_reference_class(cuda_device, ref, n, super_mode):
    """``stitch(images_dic, draw_descriptors=True)``: the reference draws its overlay at every stage (:244-245), the
    product composites once on the GPU and places each stage's overlay afterwards - the same picture."""
    h, w = 120, 200
    st, homographies, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, super_mode=super_mode, kind="smooth")
    rs = build_ref.calibrated_stitcher(ref, images, homographies, super_mode=super_mode)
    for ours, theirs in zip(st.stitchers, rs.stitchers):
        ours.sid = theirs.sid
    want = rs.stitch(images, draw_descriptors=True)
    got = st.stitch(images, draw_descriptors=True)
    assert got.shape == want.shape and np.array_equal(got, want)
    assert not np.array_equal(got, st.stitch(images))      # something was drawn


def test_cuda_shape_fixup_equals_the_reference_class(cuda_device, ref):
    """Frames that do not have the calibrated size: the reference warns and resizes them with
    ``cv2.resize(INTER_LINEAR)`` before it stitches (StitcherClass.py:226-233) - smaller and larger camera frames,
    and a first image of the wrong size; the product resizes on the GPU and ends with the same panorama."""
    import cv2
    n, h, w = 4, 120, 200
    st, homographies, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, kind="noise")
    rs = build_ref.calibrated_stitcher(ref, images, homographies)
    cases = {
        "one camera smaller": {2: (90, 150)},
        "one camera larger": {1: (150, 260)},
        "first image and last camera": {0: (96, 160), 3: (131, 217)},
        "every frame halved": {k: (60, 100) for k in range(n)},
    }
    for name, sizes in cases.items():
        frames = dict(images)
        for k, (hh, ww) in sizes.items():
            frames[labels[k]] = cv2.resize(images[labels[k]], (ww, hh), interpolation=cv2.INTER_AREA)
        want = rs.stitch(frames)
        got = st.stitch(frames)
        assert got.shape == want.shape and np.array_equal(got, want), name
