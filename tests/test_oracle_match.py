"""CPU: the numpy restatement of the matching path (oracle/match_model.py) against
cv2.BFMatcher itself, driven as StitcherClass.py:423-433 drives it."""
import cv2
import numpy as np
import pytest

from helpers import MATCH_QPC_GEOMETRIES, sum_of_squares_desc
from oracle import match_model, stitcher_ref


def cv2_knn(fa, fb):
    raw = cv2.BFMatcher(cv2.NORM_HAMMING).knnMatch(fa, fb, 2)
    idx = -np.ones((len(fa), 2), np.int32)
    dist = -np.ones((len(fa), 2), np.int32)
    for i, m in enumerate(raw):
        for j, mm in enumerate(m[:2]):
            idx[i, j] = mm.trainIdx
            dist[i, j] = int(mm.distance)
    return idx, dist, raw


def random_desc(rng, n, nbytes=32):
    return rng.integers(0, 256, size=(n, nbytes), dtype=np.uint8)


@pytest.mark.parametrize("nq,nt,nbytes", [(300, 400, 32), (64, 1000, 32), (100, 37, 64), (50, 50, 16)])
def test_knn_top2_equals_cv2(nq, nt, nbytes):
    rng = np.random.default_rng(nq * 1000 + nt)
    fa, fb = random_desc(rng, nq, nbytes), random_desc(rng, nt, nbytes)
    idx, dist = match_model.knn_top2(fa, fb)
    cidx, cdist, _ = cv2_knn(fa, fb)
    assert np.array_equal(idx, cidx)
    assert np.array_equal(dist, cdist)


def test_ties_go_to_the_lower_train_index():
    rng = np.random.default_rng(7)
    fb = random_desc(rng, 200)
    fb[150] = fb[20]          # exact duplicates: distance ties for every query
    fb[151] = fb[20]
    fb[90] = fb[3]
    fa = fb[[20, 3, 77, 150]].copy()
    fa[2, 0] ^= 0x81          # near 77
    idx, dist = match_model.knn_top2(fa, fb)
    cidx, cdist, _ = cv2_knn(fa, fb)
    assert np.array_equal(idx, cidx) and np.array_equal(dist, cdist)
    assert idx[0].tolist() == [20, 150] and dist[0].tolist() == [0, 0]
    assert idx[1].tolist() == [3, 90]
    # low-entropy descriptors: many coincident distances
    fa2 = (random_desc(rng, 120) & 0x03)
    fb2 = (random_desc(rng, 130) & 0x03)
    i2, d2 = match_model.knn_top2(fa2, fb2)
    c2, cd2, _ = cv2_knn(fa2, fb2)
    assert np.array_equal(i2, c2) and np.array_equal(d2, cd2)


def test_small_train_sets():
    rng = np.random.default_rng(11)
    fa = random_desc(rng, 10)
    one = random_desc(rng, 1)
    idx, dist = match_model.knn_top2(fa, one)
    cidx, cdist, raw = cv2_knn(fa, one)
    assert np.array_equal(idx, cidx) and np.array_equal(dist, cdist)
    assert all(len(m) == 1 for m in raw)
    keep, matches = match_model.ratio_test(idx, dist)
    assert not keep.any() and matches == []          # `len(m) == 2` fails (reference :431)
    idx0, dist0 = match_model.knn_top2(fa, np.zeros((0, 32), np.uint8))
    assert (idx0 == -1).all() and (dist0 == -1).all()


@pytest.mark.parametrize("ratio", [0.75, 0.6, 0.9, 1.0])
def test_ratio_loop_equals_reference_loop(ratio):
    rng = np.random.default_rng(5)
    fb = random_desc(rng, 500)
    fa = fb[rng.permutation(500)[:300]].copy()
    flips = rng.integers(0, 256, size=fa.shape, dtype=np.uint8) & rng.integers(0, 256, size=fa.shape, dtype=np.uint8) \
        & rng.integers(0, 256, size=fa.shape, dtype=np.uint8)
    fa ^= flips                                        # ~12 % of the bits flipped
    _, matches_ref, _ = stitcher_ref.match_keypoints(np.zeros((300, 2), np.float32), np.zeros((500, 2), np.float32),
                                                     fa, fb, ratio=ratio)[0:3]
    idx, dist, keep, matches = match_model.match(fa, fb, ratio)
    assert matches == matches_ref
    # integer form used nowhere in the product but worth pinning: 4*d0 < 3*d1 for ratio 0.75
    if ratio == 0.75:
        assert np.array_equal(keep, (idx[:, 1] >= 0) & (4 * dist[:, 0] < 3 * dist[:, 1]))


def test_orb_descriptors_of_a_synthetic_pair():
    from multicamera_stitching_b200 import synthetic
    imageB, imageA, H_true = synthetic.make_pair(360, 640, seed=3)
    orb = cv2.ORB_create(nfeatures=500)
    ka, fa = orb.detectAndCompute(imageA, None)
    kb, fb = orb.detectAndCompute(imageB, None)
    ka = np.float32([k.pt for k in ka])
    kb = np.float32([k.pt for k in kb])
    H, matches_ref, status = stitcher_ref.match_keypoints(ka, kb, fa, fb, 0.75, 3.0)
    _, _, _, matches = match_model.match(fa, fb, 0.75)
    assert matches == matches_ref and len(matches) > 50
    assert match_model.corner_error(H, H_true, 640, 360) < 3.0


def test_four_point_solver_equals_cv2():
    rng = np.random.default_rng(2)
    for _ in range(20):
        a = np.float32([[10, 20], [600, 35], [580, 400], [25, 380]]) + rng.normal(0, 5, (4, 2)).astype(np.float32)
        b = a + rng.normal(0, 20, (4, 2)).astype(np.float32)
        H = match_model.homography_from_4(a, b)
        Hc = cv2.getPerspectiveTransform(a, b)
        assert np.allclose(H, Hc, rtol=1e-6, atol=1e-8)
        assert match_model.reprojection_errors_sq(H, a, b).max() < 1e-12
    assert match_model.homography_from_4([[0, 0], [1, 1], [2, 2], [3, 3]], [[0, 0], [1, 0], [1, 1], [0, 1]]) is None


# ---------------------------------------------------------------------------
# exact restatements of the recalibration kernels (the bars of tests/test_gpu_recalib_exact.py)
def cv2_knn_l2(fa, fb, ratio):
    raw = cv2.BFMatcher(cv2.NORM_L2).knnMatch(fa, fb, 2)
    idx = -np.ones((len(fa), 2), np.int32)
    dist = -np.ones((len(fa), 2), np.float32)
    for i, m in enumerate(raw):
        for j, mm in enumerate(m[:2]):
            idx[i, j], dist[i, j] = mm.trainIdx, mm.distance
    keep = np.array([len(m) == 2 and m[0].distance < m[1].distance * ratio for m in raw], dtype=bool)
    return idx, dist, keep


def integer_desc(rng, n, dim=128):
    """Integer-valued float32 descriptors in 0..255, the form OpenCV's SIFT emits."""
    return np.minimum(255, rng.gamma(0.6, 40.0, size=(n, dim))).astype(np.uint8).astype(np.float32)


@pytest.mark.parametrize("nq,nt,dim,ratio", [(2000, 2000, 128, 0.75), (300, 257, 128, 0.8), (64, 129, 33, 0.75),
                                             (40, 2, 256, 0.9), (10, 1, 128, 0.75)])
def test_l2_restatement_equals_cv2_on_integer_descriptors(nq, nt, dim, ratio):
    rng = np.random.default_rng(nq + 31 * nt + dim)
    fb = integer_desc(rng, nt, dim)
    fa = integer_desc(rng, nq, dim)
    n_copy = min(nq, nt) // 2
    fa[:n_copy] = np.clip(fb[rng.permutation(nt)[:n_copy]] + rng.integers(-6, 7, (n_copy, dim)), 0, 255)
    if nt >= 3:                        # exact ties: equal distance, the lower train index first
        fb[nt - 1] = fb[0]
        fa[nq - 1] = fb[0]
    idx, dist, keep = match_model.l2_top2_f32(fa, fb, ratio)
    cidx, cdist, ckeep = cv2_knn_l2(fa, fb, ratio)
    assert np.array_equal(idx, cidx)
    assert np.array_equal(dist, cdist)
    assert np.array_equal(keep, ckeep)


def test_l2_ranks_by_the_rooted_distance_like_cv2():
    """Above 2^22 neighbouring integer sums share one float32 square root.  cv2 ranks the rooted distances, so the
    lower train index comes first even where its sum of squares is the larger one."""
    n = 4_200_782
    assert np.sqrt(np.float32(n)) == np.sqrt(np.float32(n + 1))
    fa = np.zeros((2, 128), np.float32)
    fa[1, 127] = 1.0                                          # (a - b)^2 sums shift, the tie stays
    fb = np.stack([sum_of_squares_desc(n + 1), sum_of_squares_desc(n), sum_of_squares_desc(n + 9000)])
    idx, dist, keep = match_model.l2_top2_f32(fa, fb, 0.75)
    cidx, cdist, ckeep = cv2_knn_l2(fa, fb, 0.75)
    assert np.array_equal(idx, cidx) and np.array_equal(dist, cdist) and np.array_equal(keep, ckeep)
    assert idx[0].tolist() == [0, 1] and dist[0, 0] == dist[0, 1]


def test_l2_ratio_boundaries_from_perfect_squares():
    fa = np.zeros((1, 8), np.float32)
    fb = np.zeros((3, 8), np.float32)
    fb[0, 0], fb[1, 3], fb[2, 5] = 4.0, 3.0, 9.0              # distances 4, 3, 9
    for ratio, kept in [(0.75, False), (0.7500001, True), (0.7499999, False)]:
        idx, dist, keep = match_model.l2_top2_f32(fa, fb, ratio)
        assert idx[0].tolist() == [1, 0] and dist[0].tolist() == [3.0, 4.0] and keep[0] == kept
        assert np.array_equal(keep, cv2_knn_l2(fa, fb, ratio)[2])


def test_four_point_restatement_equals_the_solvers():
    """``homography_4pt_exact`` (the kernel's closed form) against the 8 x 8 solve to 1e-9 relative and against
    ``cv2.getPerspectiveTransform``, whose own solve lands ~1e-8 away from both, to 1e-6; and it rejects exactly
    the samples OpenCV's checkSubset rule rejects."""
    rng = np.random.default_rng(4)
    for _ in range(200):
        a = np.float32([[10, 20], [600, 35], [580, 400], [25, 380]]) + rng.normal(0, 40, (4, 2)).astype(np.float32)
        b = a * np.float32(rng.uniform(0.5, 2.0)) + rng.normal(0, 30, (4, 2)).astype(np.float32)
        H = match_model.homography_4pt_exact(a, b)
        if not match_model.sample_is_valid(a, b):
            assert H is None
            continue
        H = H.reshape(3, 3)
        assert H[2, 2] == 1.0
        Hs = match_model.homography_from_4(a, b)
        assert np.abs(H - Hs).max() <= 1e-9 * np.abs(Hs).max()
        Hc = cv2.getPerspectiveTransform(a, b)
        assert np.abs(H - Hc).max() <= 1e-6 * np.abs(Hc).max()
        assert match_model.reprojection_errors_sq(H, a, b).max() < 1e-16
    rejected = [([[0, 0], [1, 1], [2, 2], [3, 3]], [[0, 0], [1, 0], [1, 1], [0, 1]]),          # collinear in A
                ([[0, 0], [1, 0], [1, 1], [0, 1]], [[0, 0], [0, 1], [1, 1], [1, 0]]),          # mirrored: folds
                ([[0, 0], [1, 0], [1, 1], [0, 1]], [[0, 0], [1, 0], [0, 1], [1, 1]]),          # crossed quad
                ([[0, 0], [0, 0], [1, 1], [0, 1]], [[0, 0], [1, 0], [1, 1], [0, 1]])]          # repeated point
    for a, b in rejected:
        a, b = np.float32(a), np.float32(b)
        assert not match_model.sample_is_valid(a, b) and match_model.homography_4pt_exact(a, b) is None


def test_ransac_counts_restatement_against_float64_errors():
    """The float32 inlier test agrees with the float64 reprojection error away from the threshold, and at
    threshold 0 counts exactly the correspondences that reproject without error."""
    rng = np.random.default_rng(6)
    a = rng.uniform(0, 1900, (3000, 2)).astype(np.float32)
    H = np.array([0.97, 0.02, 310.0, -0.015, 1.01, 7.5, 1e-5, -2e-5, 1.0])
    p = np.c_[a.astype(np.float64), np.ones(len(a))] @ H.reshape(3, 3).T
    b = (p[:, :2] / p[:, 2:] + rng.normal(0, 2.0, (len(a), 2))).astype(np.float32)
    count, mask = match_model.ransac_counts_f32(H, a, b, 3.0)
    err = match_model.reprojection_errors_sq(H.reshape(3, 3), a, b)
    clear = np.abs(err - 9.0) > 1e-3
    assert np.array_equal(mask[clear], err[clear] <= 9.0) and count == int(mask.sum())
    T = np.array([1.0, 0, 3, 0, 1, -5, 0, 0, 1])              # integer translation: exact in float32
    ai = rng.integers(0, 1000, (50, 2)).astype(np.float32)
    bi = ai + np.float32([3, -5])
    bi[::2, 0] += np.float32(0.5)
    count, mask = match_model.ransac_counts_f32(T, ai, bi, 0.0)
    assert count == 25 and mask[1::2].all() and not mask[::2].any()


def test_sift_descriptors_are_integers_in_0_255():
    """The premise of the L2 kernel's exactness: OpenCV's SIFT emits integer-valued floats in 0..255, so every
    square and partial sum of a 128-float descriptor is an integer below 2^24, exact in float32."""
    from multicamera_stitching_b200 import synthetic
    imageB, imageA, _ = synthetic.make_pair(360, 640, seed=3)
    sift = cv2.SIFT_create()
    for img in (imageA, imageB):
        kps, desc = sift.detectAndCompute(img, None)
        assert desc.dtype == np.float32 and desc.shape == (len(kps), 128) and len(kps) > 100
        assert np.array_equal(desc, np.round(desc)) and desc.min() >= 0 and desc.max() <= 255
        assert (desc.astype(np.int64) ** 2).sum(axis=1).max() < 2 ** 24


def test_match_qpc_paths_of_the_gpu_geometries():
    """Each queries-per-CTA path of the Hamming launcher is selected by one geometry of the GPU tests."""
    assert sorted(q for _, _, q in MATCH_QPC_GEOMETRIES) == [8, 16, 24, 32]
    for batch, nq_max, qpc in MATCH_QPC_GEOMETRIES:
        assert match_model.match_qpc(nq_max, batch) == qpc, (batch, nq_max)
    assert match_model.match_qpc(1, 65535) == 32 and match_model.match_qpc(296, 1) == 8


def test_knn_top2_large_equals_the_all_pairs_form():
    rng = np.random.default_rng(13)
    for nbytes in (16, 32, 64):
        fb = random_desc(rng, 3000, nbytes) & 0x0F               # low entropy: ties on both ranks
        fb[2999] = fb[5]
        fa = np.concatenate([fb[[5, 17, 2999]], random_desc(rng, 60, nbytes) & 0x0F])
        for m in (3000, 2, 1, 0):
            idx, dist = match_model.knn_top2_large(fa, fb[:m])
            ridx, rdist = match_model.knn_top2(fa, fb[:m])
            assert np.array_equal(idx, ridx) and np.array_equal(dist, rdist)
