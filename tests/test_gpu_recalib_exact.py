"""GPU: the recalibration kernels bit for bit against exact restatements (oracle/match_model.py).

The library is built without contraction (``--fmad=false``), so every kernel output is fully determined by its
documented order of operations: the RANSAC scorer's float64 4-point solve and float32 inlier test, its winner
(lowest index among equal maxima) and mask, the Hamming matcher's integer distances, and the L2 matcher's float32
sum (k ascending, one accumulator, then ``sqrtf``).  Every comparison here is exact, at the shapes where the
launchers switch paths: the Hamming kernel's queries per CTA and 2048-descriptor train chunks, its 21-bit train
index, the L2 kernel's 32-query / 128-train tiles and ``dim + 1`` shared-memory pitch up to ``dim = 256``, the
RANSAC select kernel's 256-stride mask loop, the 65 535-pair grid limit.  Ragged batches carry poison in their
padded rows (copies of true partners / inliers), so a kernel reading past a pair's own count changes a result."""
import cv2
import numpy as np
import pytest
import torch

from helpers import MATCH_QPC_GEOMETRIES, sum_of_squares_desc
from multicamera_stitching_b200 import StitcherBase, recalib, synthetic
from oracle import match_model, stitcher_ref

pytestmark = pytest.mark.gpu


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


# ---------------------------------------------------------------------------
# RANSAC scoring
def correspondences(n, seed, outlier_frac=0.3, w=1920, h=1080, sigma=1.0):
    rng = np.random.default_rng(seed)
    H = np.array([[0.97, 0.02, 740.3], [-0.012, 0.985, 8.1], [1.2e-5, -6e-6, 1.0]])
    a = np.stack([rng.uniform(0, w, n), rng.uniform(0, h, n)], axis=1)
    p = np.c_[a, np.ones(n)] @ H.T
    b = p[:, :2] / p[:, 2:3] + rng.normal(0, sigma, (n, 2))
    out = rng.permutation(n)[:int(outlier_frac * n)]
    b[out] = np.stack([rng.uniform(0, 2 * w, len(out)), rng.uniform(0, h, len(out))], axis=1)
    inl = np.ones(n, bool)
    inl[out] = False
    first = np.nonzero(inl)[0][:4]                              # points 0..3 are inliers: a valid first sample
    order = np.r_[first, np.setdiff1d(np.arange(n), first)]
    return a[order].astype(np.float32), b[order].astype(np.float32), inl[order]


def restate_ransac(A, B, S, thresh, n=None):
    """What ``mcs_ransac_homography`` must write: ``(counts [P,K], H_k [P,K,9], best [P], mask [P,N])``."""
    P, N, _ = A.shape
    K = S.shape[1]
    n = [N] * P if n is None else [min(int(v), N) for v in n]
    counts = -np.ones((P, K), np.int32)
    H_k = np.zeros((P, K, 9), np.float64)
    best = -np.ones(P, np.int32)
    mask = np.zeros((P, N), np.uint8)
    for i in range(P):
        a, b = A[i, :n[i]], B[i, :n[i]]
        for h in range(K):
            s = S[i, h]
            if (s < 0).any() or (s >= n[i]).any():
                continue
            H = match_model.homography_4pt_exact(a[s], b[s])
            if H is not None:
                H_k[i, h] = H
                counts[i, h] = match_model.ransac_counts_f32(H, a, b, thresh)[0]
        if (counts[i] >= 0).any():
            best[i] = int(np.argmax(counts[i]))                 # first of equal maxima; -1 never wins over >= 0
            mask[i, :n[i]] = match_model.ransac_counts_f32(H_k[i, best[i]], a, b, thresh)[1]
    return counts, H_k, best, mask


def run_ransac(A, B, S, thresh, n=None):
    counts, H_k, best, mask = recalib.ransac_batch(_dev(A), _dev(B), _dev(S.astype(np.int32)), thresh,
                                                   n=None if n is None else _dev(np.int32(n)))
    return counts.cpu().numpy(), H_k.cpu().numpy(), best.cpu().numpy(), mask.cpu().numpy()


def assert_ransac_exact(got, exp):
    counts, H_k, best, mask = got
    ecounts, eH_k, ebest, emask = exp
    assert np.array_equal(counts, ecounts), np.argwhere(counts != ecounts)[:8]
    bad = np.argwhere((H_k.view(np.uint64) != eH_k.view(np.uint64)).any(axis=-1))
    assert len(bad) == 0, bad[:8]                               # bit for bit, zeros where the sample is rejected
    assert np.array_equal(best, ebest), (best, ebest)
    assert np.array_equal(mask, emask), np.argwhere(mask != emask)[:8]


@pytest.mark.parametrize("k", [1, 7, 2001])
@pytest.mark.parametrize("n", [4, 31, 33, 257, 5000])
def test_ransac_scores_equal_the_restatement(cuda_device, n, k):
    a, b, _ = correspondences(n, seed=n + k, outlier_frac=0.3 if n > 4 else 0.0)
    S = recalib.draw_samples(n, k, seed=k).copy()[None]
    S[0, 0] = [0, 1, 2, 3]
    counts = restate_ransac(a[None], b[None], S, 3.0)[0][0]
    top = int(np.argmax(counts))
    if k > 1 and top != k - 1:                                  # a tie on the maximum, at a later index
        S[0, k - 1] = S[0, top]
    exp = restate_ransac(a[None], b[None], S, 3.0)
    assert (exp[0] >= 0).any()
    if k > 1:
        assert exp[2][0] == top < k - 1 and exp[0][0, k - 1] == exp[0][0, top]
    assert_ransac_exact(run_ransac(a[None], b[None], S, 3.0), exp)


def test_ransac_ragged_batch_with_poisoned_padding(cuda_device):
    """Pairs of 5000, 257, 33, 4 and 0 points padded to 5000; the padded points of every pair are copies of its
    true inliers, so a count or mask that looked past ``n[i]`` would change.  Half the samples index the padded
    range, some sit exactly at ``n[i]`` or below 0: those hypotheses are rejected (-1, H zero)."""
    sizes = [5000, 257, 33, 4, 0]
    N, K = max(sizes), 301
    A = np.zeros((len(sizes), N, 2), np.float32)
    B = np.zeros_like(A)
    S = np.zeros((len(sizes), K, 4), np.int32)
    for i, n in enumerate(sizes):
        a, b, inl = correspondences(N, seed=40 + i)
        A[i], B[i] = a, b
        src = np.nonzero(inl[:n])[0] if inl[:n].any() else np.nonzero(inl)[0]
        pad = np.resize(src, N - n)
        A[i, n:], B[i, n:] = a[pad], b[pad]
        S[i, :150] = recalib.draw_samples(max(n, 4), 150, seed=i)
        S[i, 150:] = recalib.draw_samples(N, K - 150, seed=100 + i)
        S[i, 0] = [0, 1, 2, 3]
        S[i, 7] = [0, 1, 2, n]
        S[i, 8] = [-1, 0, 1, 2]
    exp = restate_ransac(A, B, S, 3.0, n=sizes)
    assert (exp[0][:4] >= 0).any(axis=1).all() and (exp[0][4] == -1).all() and exp[2][4] == -1
    assert (exp[0][:, 7:9] == -1).all()
    assert_ransac_exact(run_ransac(A, B, S, 3.0, n=sizes), exp)


def test_ransac_threshold_zero_counts_exact_reprojections(cuda_device):
    """At threshold 0 a point is an inlier only if it reprojects with an error of exactly 0: the ``<=`` of
    OpenCV's test is hit on every inlier."""
    rng = np.random.default_rng(17)
    n = 400
    a = rng.integers(0, 1900, (n, 2)).astype(np.float32)
    b = a + np.float32([3, -5])
    b[::3] += rng.uniform(-2, 2, (len(b[::3]), 2)).astype(np.float32)
    S = recalib.draw_samples(n, 64, seed=2).copy()[None]
    exp = restate_ransac(a[None], b[None], S, 0.0)
    assert exp[0].max() >= 200                                  # the exact translation reprojects exactly
    assert_ransac_exact(run_ransac(a[None], b[None], S, 0.0), exp)


def test_ransac_without_hypotheses_and_all_degenerate(cuda_device):
    a, b, _ = correspondences(300, seed=5)
    got = run_ransac(a[None], b[None], np.zeros((1, 0, 4), np.int32), 3.0)
    assert got[0].shape == (1, 0) and got[2].tolist() == [-1] and not got[3].any()
    line = np.stack([np.arange(50), 2 * np.arange(50) + 1], axis=1).astype(np.float32)   # every sample collinear
    S = recalib.draw_samples(50, 200, seed=1)[None]
    exp = restate_ransac(line[None], line[None] + 7, S, 3.0)
    assert (exp[0] == -1).all() and exp[2][0] == -1
    assert_ransac_exact(run_ransac(line[None], line[None] + 7, S, 3.0), exp)


def test_find_homography_batch_equals_single_calls(cuda_device):
    a0, b0, _ = correspondences(800, seed=11)
    a1, b1, _ = correspondences(300, seed=12, outlier_frac=0.5)
    line = np.stack([np.arange(20), 3 * np.arange(20)], axis=1).astype(np.float32)
    pairs = [(a0[:3], b0[:3]), (a0, b0), (line, line + 1), (a1, b1)]
    batch = recalib.find_homography_ransac_batch(pairs, 3.0)
    for (a, b), (H, status) in zip(pairs, batch):
        H1, s1 = recalib.find_homography_ransac(a, b, 3.0)
        assert (H is None) == (H1 is None) and (status is None) == (s1 is None)
        if H is not None:
            assert np.array_equal(H, H1) and np.array_equal(status, s1)
    assert batch[0] == (None, None) and batch[2] == (None, None) and batch[1][0] is not None and batch[3][0] is not None


# ---------------------------------------------------------------------------
# matchers: ragged batches with poisoned padding
def pad_poisoned(fa_list, fb_list, rng):
    """Pads a ragged batch.  Padded train rows are copies of the pair's queries (distance 0 to them) and padded
    query rows copies of its trains, so a kernel reading past ``nt[i]`` or emitting rows past ``nq[i]`` would
    report a distance-0 partner."""
    D, dt = fa_list[0].shape[1], fa_list[0].dtype
    nq_max = max(1, max(len(f) for f in fa_list))
    nt_max = max(1, max(len(f) for f in fb_list))

    def fill(rows, src, n):
        if len(src) == 0:
            src = rng.integers(0, 256, (4, D)).astype(dt)
        rows[:] = src[np.arange(n) % len(src)]

    q = np.empty((len(fa_list), nq_max, D), dt)
    t = np.empty((len(fa_list), nt_max, D), dt)
    for i, (fa, fb) in enumerate(zip(fa_list, fb_list)):
        q[i, :len(fa)], t[i, :len(fb)] = fa, fb
        fill(q[i, len(fa):], fb, nq_max - len(fa))
        fill(t[i, len(fb):], fa, nt_max - len(fb))
    return q, t


def gpu_top2(q, t, nq=None, nt=None, ratio=0.75):
    idx2, dist2, keep = recalib.match_top2_batch(_dev(q), _dev(t), None if nq is None else _dev(np.int32(nq)),
                                                 None if nt is None else _dev(np.int32(nt)), ratio)
    return idx2.cpu().numpy(), dist2.cpu().numpy(), keep.cpu().numpy().astype(bool)


def assert_pairs_exact(got, fa_list, refs):
    idx2, dist2, keep = got
    for i, (fa, (ridx, rdist, rkeep)) in enumerate(zip(fa_list, refs)):
        n = len(fa)
        assert np.array_equal(idx2[i, :n], ridx), (i, np.argwhere(idx2[i, :n] != ridx)[:8])
        assert np.array_equal(dist2[i, :n], rdist), (i, np.argwhere(dist2[i, :n] != rdist)[:8])
        assert np.array_equal(keep[i, :n], rkeep), i
        assert (idx2[i, n:] == -1).all() and (dist2[i, n:] == -1).all() and not keep[i, n:].any(), i


def match_ragged(fa_list, fb_list, ratio, seed):
    q, t = pad_poisoned(fa_list, fb_list, np.random.default_rng(seed))
    return gpu_top2(q, t, [len(f) for f in fa_list], [len(f) for f in fb_list], ratio)


def hamming_refs(fa_list, fb_list, ratio):
    return [match_model.match(fa, fb, ratio)[:3] for fa, fb in zip(fa_list, fb_list)]


def l2_refs(fa_list, fb_list, ratio):
    return [match_model.l2_top2_f32(fa, fb, ratio) for fa, fb in zip(fa_list, fb_list)]


def planted_desc(rng, nq, nt, nbytes, partners=()):
    """Random binary descriptors; half the queries (and the given train indices) get a partner a few bits away."""
    fb = rng.integers(0, 256, (nt, nbytes), dtype=np.uint8)
    fa = rng.integers(0, 256, (nq, nbytes), dtype=np.uint8)
    extra = rng.permutation(nt)[:max(0, min(nq, nt) // 2 - len(partners))]
    tgt = np.concatenate([np.asarray(partners, np.int64), extra])[:nq]
    fa[:len(tgt)] = fb[tgt]
    fa[:len(tgt), :2] ^= rng.integers(0, 256, (len(tgt), 2), dtype=np.uint8) & 0x11
    return fa, fb


# ---------------------------------------------------------------------------
# Hamming matcher
@pytest.mark.parametrize("batch,nq_max,qpc", MATCH_QPC_GEOMETRIES)
def test_hamming_each_queries_per_cta_path(cuda_device, batch, nq_max, qpc):
    assert match_model.match_qpc(nq_max, batch) == qpc
    rng = np.random.default_rng(qpc)
    sizes = [(nq_max, 700)] + [(nq_max - 37 * j, 700 - 101 * j) for j in range(1, batch)]
    pairs = [planted_desc(rng, nq, nt, 32) for nq, nt in sizes]
    fa_list, fb_list = [p[0] for p in pairs], [p[1] for p in pairs]
    assert_pairs_exact(match_ragged(fa_list, fb_list, 0.75, seed=qpc), fa_list, hamming_refs(fa_list, fb_list, 0.75))


@pytest.mark.parametrize("nbytes", [16, 32, 64])
def test_hamming_train_chunk_boundaries(cuda_device, nbytes):
    """Train counts around the 2048-descriptor shared-memory chunk, partners planted on both sides of each
    boundary, in one ragged batch (and the largest pair alone, without count arrays)."""
    rng = np.random.default_rng(nbytes)
    nts = [2047, 2048, 2049, 4096, 4097]
    edges = [0, 2046, 2047, 2048, 4095, 4096]
    pairs = [planted_desc(rng, 300, nt, nbytes, [e for e in edges if e < nt]) for nt in nts]
    fa_list, fb_list = [p[0] for p in pairs], [p[1] for p in pairs]
    refs = hamming_refs(fa_list, fb_list, 0.75)
    assert_pairs_exact(match_ragged(fa_list, fb_list, 0.75, seed=nbytes), fa_list, refs)
    assert_pairs_exact(gpu_top2(fa_list[-1][None], fb_list[-1][None]), fa_list[-1:], refs[-1:])


@pytest.mark.parametrize("nbytes", [16, 32, 64])
def test_hamming_distance_zero_and_maximum(cuda_device, nbytes):
    rng = np.random.default_rng(3 + nbytes)
    x = rng.integers(0, 256, (1, nbytes), dtype=np.uint8)
    fb = np.repeat(x, 40, axis=0)                               # every train equal: ties everywhere
    fa = np.concatenate([x, ~x, x ^ 1])
    ref = match_model.match(fa, fb, 0.75)[:3]
    assert ref[1][1].tolist() == [8 * nbytes, 8 * nbytes] and ref[1][0].tolist() == [0, 0]
    assert ref[0].tolist() == [[0, 1]] * 3
    assert_pairs_exact(gpu_top2(fa[None], fb[None]), [fa], [ref])


def test_hamming_train_index_above_2_to_the_20(cuda_device):
    """nt = 2^21 - 1, the largest train set the 21-bit index of the packed key holds (64 MB of 32-byte
    descriptors); some queries' true partners sit above index 2^20.  Reference: ``knn_top2_large``, the
    query-at-a-time form of the restatement (the all-pairs matrix would take 16 GB here)."""
    nt = (1 << 21) - 1
    rng = np.random.default_rng(21)
    fb = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    partners = [nt - 1, nt - 2, 1 << 20, (1 << 20) + 1, (1 << 20) - 1, 1_500_000, 12]
    fa = rng.integers(0, 256, (40, 32), dtype=np.uint8)
    fa[:len(partners)] = fb[partners]
    fa[:len(partners), 0] ^= 0x01
    fb[nt - 3] = fb[nt - 2]                                     # a tie on the best, decided by the index
    ridx, rdist = match_model.knn_top2_large(fa, fb)
    rkeep = match_model.ratio_test(ridx, rdist, 0.75)[0]
    assert ridx[:len(partners), 0].tolist() == [partners[0], nt - 3] + partners[2:] and ridx[1, 1] == nt - 2
    assert_pairs_exact(gpu_top2(fa[None], fb[None]), [fa], [(ridx, rdist, rkeep)])


def test_hamming_65535_tiny_pairs(cuda_device):
    """The largest batch the grid's y dimension holds, ragged (0..3 queries, 0..5 trains per pair)."""
    rng = np.random.default_rng(65535)
    B = 65535
    nq = rng.integers(0, 4, B)
    nt = rng.integers(0, 6, B)
    fa_list = [rng.integers(0, 256, (a, 16), dtype=np.uint8) & 0x0F for a in nq]
    fb_list = [rng.integers(0, 256, (b, 16), dtype=np.uint8) & 0x0F for b in nt]
    got = match_ragged(fa_list, fb_list, 0.8, seed=1)
    assert_pairs_exact(got, fa_list, hamming_refs(fa_list, fb_list, 0.8))


def bits_desc(lo, hi, nbytes=32):
    """A binary descriptor with bits lo .. hi - 1 set."""
    d = np.zeros(nbytes * 8, np.uint8)
    d[lo:hi] = 1
    return np.packbits(d)


@pytest.mark.parametrize("ratio,kept", [(0.75, False), (0.7500001, True), (0.7499999, False)])
def test_hamming_ratio_boundaries(cuda_device, ratio, kept):
    """Distances 3 and 4, and 6 and 8, sit exactly on ``d0 < d1 * 0.75``."""
    fa = np.stack([bits_desc(0, 0), bits_desc(128, 138)])
    fb = np.stack([bits_desc(0, 7), bits_desc(0, 4), bits_desc(0, 3), bits_desc(128, 132), bits_desc(128, 146)])
    ref = match_model.match(fa, fb, ratio)[:3]
    assert ref[1].tolist() == [[3, 4], [6, 8]] and ref[2].tolist() == [kept, kept]
    assert_pairs_exact(gpu_top2(fa[None], fb[None], ratio=ratio), [fa], [ref])


# ---------------------------------------------------------------------------
# L2 matcher
def wide_floats(rng, shape):
    """Signed magnitudes from 1e-25 to 1e15 (denormal and underflowing squares, no overflow), some exact zeros."""
    x = rng.choice([-1.0, 1.0], shape) * 10.0 ** rng.uniform(-25, 15, shape)
    x[rng.random(shape) < 0.05] = 0.0
    return x.astype(np.float32)


@pytest.mark.parametrize("kind", ["normal", "wide"])
def test_l2_general_floats(cuda_device, kind):
    rng = np.random.default_rng(7 if kind == "normal" else 8)
    make = (lambda s: rng.normal(0, 1, s).astype(np.float32)) if kind == "normal" else (lambda s: wide_floats(rng, s))
    fb = make((1500, 128))
    fa = make((1000, 128))
    fa[:400] = fb[rng.permutation(1500)[:400]] * np.float32(1.001)
    ref = match_model.l2_top2_f32(fa, fb, 0.8)
    assert ref[2].sum() > 100
    assert_pairs_exact(gpu_top2(fa[None], fb[None], ratio=0.8), [fa], [ref])


@pytest.mark.parametrize("dim", [1, 2, 3, 33, 127, 129, 255, 256])
def test_l2_tile_boundaries(cuda_device, dim):
    """Every (nq, nt) of {31, 32, 33} x {127, 128, 129, 255, 256, 257} around the 32-query and 128-train tiles,
    in one poisoned ragged batch, at dims around the ``dim + 1`` pitch up to the 164 480 B of ``dim = 256``."""
    rng = np.random.default_rng(dim)
    sizes = [(a, b) for a in (31, 32, 33) for b in (127, 128, 129, 255, 256, 257)]
    fb_list = [rng.normal(0, 1, (b, dim)).astype(np.float32) for _, b in sizes]
    fa_list = [np.concatenate([fb[rng.permutation(len(fb))[:a // 2]] + rng.normal(0, 0.1, (a // 2, dim)),
                               rng.normal(0, 1, (a - a // 2, dim))]).astype(np.float32)
               for (a, _), fb in zip(sizes, fb_list)]
    refs = l2_refs(fa_list, fb_list, 0.75)
    assert_pairs_exact(match_ragged(fa_list, fb_list, 0.75, seed=dim), fa_list, refs)
    assert_pairs_exact(gpu_top2(fa_list[-1][None], fb_list[-1][None]), fa_list[-1:], refs[-1:])


def test_l2_65535_tiny_pairs(cuda_device):
    rng = np.random.default_rng(65536)
    B, D = 65535, 5
    nq = rng.integers(0, 4, B)
    nt = rng.integers(0, 6, B)
    Q = rng.integers(0, 4, (B, 3, D)).astype(np.float32)       # small integers: many exact ties
    T = rng.integers(0, 4, (B, 5, D)).astype(np.float32)
    fa_list = [Q[i, :nq[i]] for i in range(B)]
    fb_list = [T[i, :nt[i]] for i in range(B)]
    got = match_ragged(fa_list, fb_list, 0.8, seed=2)
    refs = [None] * B
    for a in range(4):                                          # the restatement, batched by shape
        for b in range(6):
            sel = np.nonzero((nq == a) & (nt == b))[0]
            ridx, rdist, rkeep = match_model.l2_top2_f32(Q[sel, :a], T[sel, :b], 0.8)
            for j, i in enumerate(sel):
                refs[i] = (ridx[j], rdist[j], rkeep[j])
    assert_pairs_exact(got, fa_list, refs)


@pytest.mark.parametrize("ratio,kept", [(0.75, False), (0.7500001, True), (0.7499999, False)])
def test_l2_ratio_boundaries_from_perfect_squares(cuda_device, ratio, kept):
    fa = np.zeros((2, 16), np.float32)
    fa[1, 10] = 100.0
    fb = np.zeros((5, 16), np.float32)
    fb[0, 0], fb[1, 3], fb[2, 5] = 4.0, 3.0, 9.0                # query 0: distances 4, 3, 9
    fb[3:, 10] = 100.0
    fb[3, 11], fb[4, 12] = 6.0, 8.0                             # query 1: distances 6, 8
    ref = match_model.l2_top2_f32(fa, fb, ratio)
    assert ref[1].tolist() == [[3.0, 4.0], [6.0, 8.0]] and ref[2].tolist() == [kept, kept]
    assert_pairs_exact(gpu_top2(fa[None], fb[None], ratio=ratio), [fa], [ref])


def test_l2_ranks_by_the_rooted_distance(cuda_device):
    """Sums of squares 4200783 and 4200782 share one float32 square root: the lower train index comes first, as in
    cv2, although its sum is the larger."""
    fa = np.zeros((2, 128), np.float32)
    fa[1, 127] = 1.0
    fb = np.stack([sum_of_squares_desc(n) for n in (4_200_783, 4_200_782, 4_209_782)])
    ref = match_model.l2_top2_f32(fa, fb, 0.75)
    assert ref[0][0].tolist() == [0, 1] and ref[1][0, 0] == ref[1][0, 1]
    raw = cv2.BFMatcher(cv2.NORM_L2).knnMatch(fa, fb, 2)
    assert ref[0].tolist() == [[m[0].trainIdx, m[1].trainIdx] for m in raw]
    assert_pairs_exact(gpu_top2(fa[None], fb[None]), [fa], [ref])


# ---------------------------------------------------------------------------
def test_match_keypoints_on_real_sift_features(cuda_device):
    """``StitcherBase.matchKeypoints`` with the reference's own detector (``descriptor = "SIFT"``) on a synthetic
    pair: the match list equals the reference loop's, the homography agrees at the frame corners."""
    imageB, imageA, H_true = synthetic.make_pair(540, 960, seed=5)
    sb = StitcherBase()
    sb.descriptor = "SIFT"
    kpsA, fa = sb.detectAndDescribe(imageA)
    kpsB, fb = sb.detectAndDescribe(imageB)
    assert fa.dtype == np.float32 and fa.shape[1] == 128
    H, matches, status = sb.matchKeypoints(kpsA, kpsB, fa, fb, ratio=0.75, reprojThresh=3.0)
    Hr, matches_ref, status_ref = stitcher_ref.match_keypoints(kpsA, kpsB, fa, fb, 0.75, 3.0)
    assert matches == matches_ref and len(matches) > 50
    assert status.shape == status_ref.shape
    assert match_model.corner_error(H, Hr, 960, 540) < 0.5
    assert match_model.corner_error(H, H_true, 960, 540) < 2.5
