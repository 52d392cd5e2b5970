"""Pins ``oracle/stitcher_ref.py`` against the REFERENCE'S OWN ``StitcherClass.py``, run here.

``oracle/build_ref.py`` makes ``/root/reference/PostScripts/Stitcher/StitcherClass.py`` importable under Python 3
with a four-line mechanical patch list (indentation of ``__str__``, a dict view, the OpenCV-version switch of the
feature detector) and imports the reference's ``Utils.py`` unchanged.  Every function of the oracle is held against
the reference method it restates (SURVEY.md section 8 rows a1-a5, a7), on the seeded synthetic inputs of the other
tests: same state fields, same panoramas, same match lists, bit for bit.

CPU only.  A test that needs the reference's class is skipped where neither the reference tree nor its build output
``oracle/_ref`` is present (a clean checkout): the repository does not ship the reference.  What runs there of it is
the committed fixture ``tests/golden/chain_ref.npz`` (tests/test_golden.py), generated from the reference classes by
``scripts/make_golden.py``: the panoramas and canvas geometry of three chains, not the other comparisons made here.
The product-side halves of the fallback checks below need no reference and always run.
"""
import os
import pickle

import cv2
import numpy as np
import pytest

from helpers import synthetic_chain
from multicamera_stitching_b200 import synthetic
from oracle import build_ref, stitcher_ref


FIELDS = ("cachedAH", "cachedAINVH", "cachedBH", "cachedBINVH", "Bpts", "Apts", "ABSize", "x_limits", "y_limits",
          "AimgSize", "BimgSize")


@pytest.fixture(scope="module")
def ref_or_none():
    """The reference module, or None where neither the reference tree nor oracle/_ref is present."""
    return build_ref.load()


@pytest.fixture(scope="module")
def ref(ref_or_none):
    if ref_or_none is None:
        pytest.skip("reference not present (neither the reference tree nor oracle/_ref)")
    return ref_or_none


def inject_homography(sb, H):
    """Makes ``StitcherBase.calibrate`` (StitcherClass.py:258-354) run its REAL geometry code on a given homography:
    only the feature detection and matching in front of it are replaced."""
    sb.detectAndDescribe = lambda image: (np.zeros((1, 2), np.float32), None)
    sb.matchKeypoints = lambda **kw: (np.array(H, dtype=np.float64), [(0, 0)] * 5, np.ones((5, 1), np.uint8))


def assert_state_equal(ref_sb, st):
    for f in FIELDS:
        a, b = getattr(ref_sb, f), st[f]
        assert (a is None) == (b is None), f
        if a is not None:
            a, b = np.asarray(a), np.asarray(b)
            assert a.dtype.kind == b.dtype.kind and a.shape == b.shape and np.array_equal(a, b), f


def random_homographies(n, h, w, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        ang = rng.uniform(-0.2, 0.2)
        s = rng.uniform(0.7, 1.3)
        H = np.array([[s * np.cos(ang), -s * np.sin(ang) + rng.uniform(-0.05, 0.05), rng.uniform(-0.3, 0.9) * w],
                      [s * np.sin(ang), s * np.cos(ang) * rng.uniform(0.9, 1.1), rng.uniform(-0.4, 0.4) * h],
                      [rng.uniform(-2e-4, 2e-4), rng.uniform(-2e-4, 2e-4), 1.0]])
        out.append(H)
    return out


# ---- a4: canvas geometry (StitcherClass.py:293-351) ------------------------------------------------
@pytest.mark.parametrize("offsets", [(0, 0), (3, 5), (10, 10), (-7, 4)])
def test_geometry_equals_reference_calibrate(ref, offsets):
    h, w = 90, 160
    imageA = synthetic.make_frame(h, w, 3, 1, 0, "noise")
    imageB = synthetic.make_frame(h + 12, w - 20, 3, 0, 0, "noise")
    homs = [synthetic.make_homography(k, h, w, w - 20) for k in range(4)]
    homs += [synthetic.homography_from_points(h, w, w - 20)] + random_homographies(24, h, w, seed=11)
    for H in homs:
        sb = ref.StitcherBase(sid="pin", super_mode=False)
        inject_homography(sb, H)
        sb.calibrate(images=(imageB, imageA), ratio=0.75, reprojThresh=3.0, xoffset=offsets[0], yoffset=offsets[1])
        st = stitcher_ref.new_state("pin", False)
        try:
            stitcher_ref.geometry_from_homography(st, H, imageA.shape, imageB.shape, offsets[0], offsets[1])
        except ValueError:
            # max()/min() of an empty list in the ROI limits (:344-351): the reference raises the same
            # way inside calibrate, so it never got this far
            pytest.fail("the reference accepted a homography the oracle rejects")
        assert_state_equal(sb, st)


@pytest.mark.parametrize("offsets", [(0, 0), (10, 10), (-7, 4)])
@pytest.mark.parametrize("super_mode", [False, True])
def test_product_geometry_equals_reference_calibrate(ref, offsets, super_mode):
    """The PRODUCT's own host-side geometry (``StitcherBase.set_homography`` / ``_geometry``, what the plan is built
    from) against the reference's ``calibrate`` directly, not through the oracle: every state field equal."""
    from multicamera_stitching_b200 import StitcherBase
    h, w = 90, 160
    imageA = synthetic.make_frame(h, w, 3, 1, 0, "noise")
    imageB = synthetic.make_frame(h + 12, w - 20, 3, 0, 0, "noise")
    homs = [synthetic.make_homography(k, h, w, w - 20) for k in range(4)]
    homs += [synthetic.homography_from_points(h, w, w - 20)] + random_homographies(24, h, w, seed=23)
    for H in homs:
        sb = ref.StitcherBase(sid="pin", super_mode=super_mode)
        inject_homography(sb, H)
        sb.calibrate(images=(imageB, imageA), ratio=0.75, reprojThresh=3.0, xoffset=offsets[0], yoffset=offsets[1])
        ours = StitcherBase(sid="pin", super_mode=super_mode)
        ours.set_homography(np.array(H, dtype=np.float64), shapeA=imageA.shape, shapeB=imageB.shape,
                            xoffset=offsets[0], yoffset=offsets[1])
        assert_state_equal(sb, {f: getattr(ours, f) for f in FIELDS})


# ---- a1: pair stitch (StitcherClass.py:211-256) ----------------------------------------------------
@pytest.mark.parametrize("super_mode", [False, True])
@pytest.mark.parametrize("kind", ["noise", "smooth"])
def test_stitch_pair_equals_reference(ref, super_mode, kind):
    h, w = 120, 200
    imageB = synthetic.make_frame(h, w, 3, 0, 0, kind)
    imageA = synthetic.make_frame(h, w, 3, 1, 0, kind)
    for k, H in enumerate([synthetic.make_homography(0, h, w, w), synthetic.make_homography(1, h, w, w)] +
                          random_homographies(6, h, w, seed=5)):
        sb = ref.StitcherBase(sid="p%d" % k, super_mode=super_mode)
        inject_homography(sb, H)
        sb.calibrate(images=(imageB, imageA), xoffset=2, yoffset=3)
        st = stitcher_ref.new_state("p%d" % k, super_mode)
        stitcher_ref.geometry_from_homography(st, H, imageA.shape, imageB.shape, 2, 3)
        want = sb.stitch(images=(imageB, imageA))
        got = stitcher_ref.stitch_pair(st, (imageB, imageA))
        assert want.shape == got.shape and np.array_equal(want, got)
        # frames of another size take the resize branch (:226-233)
        smallB, bigA = imageB[::2, ::2].copy(), cv2.resize(imageA, (w + 31, h + 17))
        want = sb.stitch(images=(smallB, bigA))
        got = stitcher_ref.stitch_pair(st, (smallB, bigA))
        assert want.shape == got.shape and np.array_equal(want, got)


def test_uncalibrated_pair_returns_image_b(ref_or_none):
    """An uncalibrated pair hands image B back (:255-256); the reference's side is checked where it is present."""
    imageB = synthetic.make_frame(40, 50, 3, 0, 0, "noise")
    imageA = synthetic.make_frame(40, 50, 3, 1, 0, "noise")
    if ref_or_none is not None:
        assert ref_or_none.StitcherBase().stitch((imageB, imageA)) is imageB
    assert stitcher_ref.stitch_pair(stitcher_ref.new_state(), (imageB, imageA)) is imageB


# ---- a2 / a7: the chain (StitcherClass.py:52-75, 77-112, 114-136) -----------------------------------
def reference_chain(ref, images, homographies, super_mode):
    """The reference's own ``Stitcher``, calibrated by its own ``calibrate_stitcher`` with the given stage
    homographies in place of matched features (every stage calibrates against the stitched canvas so far)."""
    rs = ref.Stitcher(images, super_mode=super_mode)
    for sb, H in zip(rs.stitchers, homographies):
        inject_homography(sb, H)
    rs.calibrate_stitcher(images, save=False)
    return rs


@pytest.mark.parametrize("n,h,w,super_mode,kind", [
    (3, 720, 1280, False, "smooth"),     # BASELINE config 1
    (3, 96, 128, False, "noise"),
    (6, 135, 240, False, "noise"),
    (4, 90, 160, True, "noise"),
    (8, 108, 192, False, "smooth"),
])
def test_chain_equals_reference_stitcher(ref, n, h, w, super_mode, kind):
    st, states, labels, images = synthetic_chain(n, h, w, 3, super_mode=super_mode, kind=kind)
    homs = []   # the homographies synthetic_chain used: they depend on the running canvas width
    cw = w
    for k in range(n - 1):
        homs.append(synthetic.make_homography(k, h, w, cw))
        cw = st.stitchers[k].result_shape()[1]
    rs = reference_chain(ref, images, homs, super_mode)
    assert list(rs.img_labels) == list(labels) == stitcher_ref.sorted_labels(images)
    assert list(rs.stitcher_labels) == stitcher_ref.stitcher_labels(labels)
    for sb, s in zip(rs.stitchers, states):
        assert_state_equal(sb, s)
    want = rs.stitch(images)
    got = stitcher_ref.stitch_chain(states, labels, images)
    assert want.shape == got.shape and np.array_equal(want, got)
    # and the product class carries the same state (same field names, StitcherClass.py:190-209)
    for sb, ours in zip(rs.stitchers, st.stitchers):
        for f in ("cachedAH", "Bpts", "ABSize", "x_limits", "y_limits", "AimgSize", "BimgSize"):
            assert np.array_equal(np.asarray(getattr(sb, f)), np.asarray(getattr(ours, f))), f
    # fewer images than labels: the reference hands back the last image (:124-128)
    fewer = {l: images[l] for l in labels[1:]}
    assert rs.stitch(fewer) is fewer[labels[-1]]
    assert stitcher_ref.stitch_chain(states, labels, fewer) is fewer[labels[-1]]


def test_random_chains_equal_reference(ref):
    """The fuzz geometry of tests/test_gpu_fuzz.py (rotation, perspective, mirrored cameras) through the reference."""
    h, w = 72, 110
    for seed in range(8):
        n = 3 + seed % 3
        images = synthetic.make_frames(n, h, w, 3, frame_index=seed, kind="noise")
        labels = stitcher_ref.sorted_labels(images)
        homs = random_homographies(n - 1, h, w, seed=100 + seed)
        try:
            rs = reference_chain(ref, images, homs, False)
        except ValueError:
            # the reference's ROI limits (:344-351) take max()/min() of lists that may be empty: it raises
            with pytest.raises(ValueError):
                stitcher_ref.calibrate_chain_from_homographies([images[l].shape for l in labels], homs)
            continue
        states = stitcher_ref.calibrate_chain_from_homographies([images[l].shape for l in labels], homs)
        for sb, s in zip(rs.stitchers, states):
            assert_state_equal(sb, s)
        assert np.array_equal(rs.stitch(images), stitcher_ref.stitch_chain(states, labels, images))


@pytest.mark.parametrize("super_mode", [False, True])
def test_random_chains_sweep_equals_reference(ref, super_mode):
    """A wider seeded sweep of the same fuzz geometry - 2 to 6 cameras, odd frame sizes, super mode, calibration
    offsets - states and panoramas equal to the reference's, or both sides refusing the geometry alike."""
    compared = 0
    for seed in range(40):
        rng = np.random.default_rng(7000 + seed)
        n = int(rng.integers(2, 7))
        h, w = int(rng.integers(40, 100)), int(rng.integers(50, 140))
        images = synthetic.make_frames(n, h, w, 3, frame_index=seed, kind="noise")
        labels = stitcher_ref.sorted_labels(images)
        homs = random_homographies(n - 1, h, w, seed=500 + seed)
        shapes = [images[l].shape for l in labels]
        try:
            rs = reference_chain(ref, images, homs, super_mode)
        except (ValueError, cv2.error) as e:
            with pytest.raises(type(e)):
                states = stitcher_ref.calibrate_chain_from_homographies(shapes, homs, super_mode=super_mode)
                stitcher_ref.stitch_chain(states, labels, images)
            continue
        states = stitcher_ref.calibrate_chain_from_homographies(shapes, homs, super_mode=super_mode)
        for sb, s in zip(rs.stitchers, states):
            assert_state_equal(sb, s)
        try:
            want = rs.stitch(images)
        except (ValueError, cv2.error) as e:
            with pytest.raises(type(e)):
                stitcher_ref.stitch_chain(states, labels, images)
            continue
        got = stitcher_ref.stitch_chain(states, labels, images)
        assert got.shape == want.shape and np.array_equal(got, want), seed
        compared += 1
    assert compared >= 20, compared


# ---- a5: matchKeypoints (StitcherClass.py:405-448), the reference's own float / L2 branch -----------------
def test_match_keypoints_equals_reference(ref):
    rng = np.random.default_rng(3)
    nA, nB = 260, 300
    featB = rng.normal(0, 40, (nB, 128)).clip(0, 255).astype(np.float32)
    perm = rng.permutation(nB)[:nA]
    featA = featB[perm] + rng.normal(0, 6, (nA, 128)).astype(np.float32)
    featA[200:] = rng.normal(0, 40, (60, 128)).clip(0, 255).astype(np.float32)   # no partner: the ratio test drops most
    H_true = np.array([[0.97, 0.02, 31.0], [-0.015, 1.01, 7.5], [1e-5, -2e-5, 1.0]])
    kpsA = rng.uniform(0, 600, (nA, 2)).astype(np.float32)
    proj = np.c_[kpsA, np.ones(nA)] @ H_true.T
    kpsB = np.zeros((nB, 2), np.float32)
    kpsB[perm] = (proj[:, :2] / proj[:, 2:]).astype(np.float32) + rng.normal(0, 0.3, (nA, 2)).astype(np.float32)
    sb = ref.StitcherBase()
    H0, m0, s0 = sb.matchKeypoints(kpsA=kpsA, kpsB=kpsB, featuresA=featA, featuresB=featB, ratio=0.75, reprojThresh=3.0)
    H1, m1, s1 = stitcher_ref.match_keypoints(kpsA, kpsB, featA, featB, ratio=0.75, reprojThresh=3.0)
    assert m0 == m1 and len(m0) > 150
    assert np.array_equal(H0, H1) and np.array_equal(s0, s1)
    # four matches or fewer: no homography (:436)
    H0, m0, s0 = sb.matchKeypoints(kpsA=kpsA[:3], kpsB=kpsB, featuresA=featA[:3], featuresB=featB)
    H1, m1, s1 = stitcher_ref.match_keypoints(kpsA[:3], kpsB, featA[:3], featB)
    assert H0 is None and H1 is None and m0 == m1 and s0 is None and s1 is None


# ---- a7: persistence (StitcherClass.py:138-177, 485-505) -------------------------------------------------
def test_reference_pickle_loads_into_the_product_class(ref, tmp_path):
    """A configuration saved by the reference's own ``save_stitcher`` (pickle of the reference object, matrices as
    lists of row arrays) loads through the product's ``load_stitcher`` with every field intact."""
    from multicamera_stitching_b200 import Stitcher
    st, states, labels, images = synthetic_chain(3, 96, 128, 3, kind="noise")
    homs, cw = [], 128
    for k in range(2):
        homs.append(synthetic.make_homography(k, 96, 128, cw))
        cw = st.stitchers[k].result_shape()[1]
    rs = reference_chain(ref, images, homs, False)
    for sb in rs.stitchers:   # the injected lambdas are test scaffolding, not state
        del sb.detectAndDescribe, sb.matchKeypoints
    path = os.path.join(str(tmp_path), "Stitcher_config.pkl")
    rs.save_stitcher(path)
    assert os.path.getsize(path) > 0
    with open(path, "rb") as f:
        head = f.read(64)
    assert b"StitcherClass_ref" in head or b"Stitcher" in pickle.dumps(rs)[:200]
    loaded = Stitcher(images).load_stitcher(path)
    assert list(loaded.img_labels) == list(labels)
    for sb, ours in zip(rs.stitchers, loaded.stitchers):
        for f in ("cachedAH", "Bpts", "ABSize", "x_limits", "y_limits", "AimgSize", "BimgSize", "super_mode", "sid"):
            assert np.array_equal(np.asarray(getattr(sb, f)), np.asarray(getattr(ours, f))), f


# ---- debug overlay (StitcherClass.py:244-245, 450-483) ----------------------------------------------------
@pytest.mark.parametrize("n,super_mode", [(3, False), (4, True), (5, False)])
def test_per_stage_overlays_equal_the_reference(ref, n, super_mode):
    """``Stitcher.stitch(draw_descriptors=True)``: the reference draws at EVERY stage; the product composites
    once and then puts each stage's overlay where its canvas ended up - same pixels.  (Host code: the panorama
    under the overlays comes from the oracle here, on the GPU it comes from the kernel.)"""
    h, w = 120, 200
    st, states, labels, images = synthetic_chain(n, h, w, 3, super_mode=super_mode, kind="smooth")
    homs, cw = [], w
    for k in range(n - 1):
        homs.append(synthetic.make_homography(k, h, w, cw))
        cw = st.stitchers[k].result_shape()[1]
    rs = reference_chain(ref, images, homs, super_mode)
    want = rs.stitch(images, draw_descriptors=True)
    base = stitcher_ref.stitch_chain(states, labels, images).copy()
    for ours, theirs in zip(st.stitchers, rs.stitchers):
        ours.sid = theirs.sid
    flat = st.plan.__func__  # noqa: F841  (the plan needs a device; the overlay code only needs the flat layers)
    from multicamera_stitching_b200 import plan as planmod
    flat = planmod.flatten_chain(st.stitchers, [images[l].shape for l in labels])

    class _P(object):
        pass
    p = _P()
    p.flat = flat
    st.plan = lambda shapes, device=None: p
    got = st._draw_overlays(base, [images[l] for l in labels])
    assert got.shape == want.shape and np.array_equal(got, want)


@pytest.mark.skipif(not build_ref.available(), reason="reference tree not present")
def test_prebuilt_reference_runs_without_the_reference_tree(tmp_path):
    """The build output (oracle/_ref: the patched class, the logging stand-in, a byte copy of the reference's
    Utils.py) is all the GPU box has: with the reference tree out of reach, ``build_ref.load()`` falls back to it
    and the reference's own ``Stitcher`` still produces the panorama of the restatement - this is the CPU arm of
    ``bench.py --impl reference`` there."""
    import subprocess
    import sys
    assert build_ref.build() is not None
    with open(os.path.join(build_ref.REF_UTILS_DIR, "Utils.py"), "rb") as f, \
            open(os.path.join(build_ref.OUT_DIR, "Calibration_Utils", "Utils.py"), "rb") as g:
        assert f.read() == g.read()
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import numpy as np\n"
        "from helpers import synthetic_chain\n"
        "from multicamera_stitching_b200 import synthetic\n"
        "from oracle import build_ref, stitcher_ref\n"
        "assert not build_ref.available() and build_ref.prebuilt()\n"
        "ref = build_ref.load()\n"
        "st, hs, labels, images = synthetic.synthetic_stitcher(4, 90, 160, 3, kind='noise')\n"
        "states = stitcher_ref.calibrate_chain_from_homographies([images[l].shape for l in labels], hs)\n"
        "rs = build_ref.calibrated_stitcher(ref, images, hs)\n"
        "assert np.array_equal(rs.stitch(images), stitcher_ref.stitch_chain(states, labels, images))\n"
        "print('prebuilt ok')\n" % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                    os.path.dirname(os.path.abspath(__file__))))
    env = dict(os.environ, MCS_REFERENCE_ROOT=str(tmp_path / "no_reference_here"))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=300)
    assert r.returncode == 0 and b"prebuilt ok" in r.stdout, r.stdout.decode(errors="replace")


def test_product_lifecycle_equals_reference(ref):
    """a7 directly against the reference objects: labels, ``__str__``, ``params_to_list`` / ``params_to_array``
    round trip and ``reset`` leave the product's stages in the state the reference's are in."""
    from multicamera_stitching_b200 import Stitcher
    h, w, n = 72, 110, 4
    images = synthetic.make_frames(n, h, w, 3, frame_index=2, kind="noise")
    labels = stitcher_ref.sorted_labels(images)
    homs = [synthetic.make_homography(k, h, w, w) for k in range(n - 1)]
    rs = reference_chain(ref, images, homs, False)
    ours = Stitcher(images)
    ours.calibrate_from_homographies([images[l].shape for l in labels], homs, xoffset=0, yoffset=0)   # :102-103
    assert list(ours.img_labels) == list(rs.img_labels) and list(ours.stitcher_labels) == list(rs.stitcher_labels)
    for a, b in zip(rs.stitchers, ours.stitchers):
        assert a.sid == b.sid
        assert str(a).split("| Matches:")[0] == str(b).split("| Matches:")[0]          # the injected calibration
        assert str(a).split("StitcherSize:")[1] == str(b).split("StitcherSize:")[1]   # carries stand-in matches
        a.params_to_list()
        b.params_to_list()
        for f in ("cachedAH", "cachedAINVH", "cachedBH", "cachedBINVH"):
            assert type(getattr(a, f)) is type(getattr(b, f)) is list
            assert np.array_equal(np.asarray(getattr(a, f)), np.asarray(getattr(b, f)))
        a.params_to_array()
        b.params_to_array()
        assert_state_equal(a, {f: getattr(b, f) for f in FIELDS})
        a.reset()
        b.reset()
        for f in FIELDS + ("matches", "status"):
            assert getattr(a, f) is None and getattr(b, f) is None, f
        assert str(a) == str(b)


def test_product_fallbacks_equal_reference(ref_or_none):
    """The frame path never raises (SURVEY section 8 b): an uncalibrated chain hands the first image through
    (:255-256), a dictionary with fewer images than labels hands back the last label's image (:124-128) - the
    product returns the very objects the reference returns, without touching a device.  The product's side always
    runs; the reference's side where it is present."""
    from multicamera_stitching_b200 import Stitcher
    images = synthetic.make_frames(3, 48, 64, 3, frame_index=0, kind="noise")
    ours = Stitcher(images)
    rs = None if ref_or_none is None else ref_or_none.Stitcher(images, super_mode=False)
    sides = [ours] if rs is None else [rs, ours]
    labels = list(ours.img_labels)
    if rs is not None:
        assert list(rs.img_labels) == labels
    for side in sides:
        assert side.stitch(images) is images[labels[0]]
        short = {l: images[l] for l in labels[1:]}                 # one image missing: the last label's image comes back
        assert side.stitch(short) is images[labels[-1]]
        short = {l: images[l] for l in labels[:2]}                 # the last label itself missing: both look it up
        with pytest.raises(KeyError):
            side.stitch(short)
        short = {labels[-1]: images[labels[-1]]}
        assert side.stitch(short) is images[labels[-1]]
        b, a = images[labels[0]], images[labels[1]]
        assert side.stitchers[0].stitch((b, a)) is b
