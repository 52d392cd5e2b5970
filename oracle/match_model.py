"""ORACLE (test infrastructure, never imported by the product package).

Transparent numpy restatement of the descriptor-matching half of
``StitcherBase.matchKeypoints`` (reference PostScripts/Stitcher/
StitcherClass.py:405-448) for binary descriptors:

  :423-424  ``matcher.knnMatch(featuresA, featuresB, 2)``  - brute force, query =
            featuresA, train = featuresB, Hamming norm for uint8 (ORB) descriptors
  :428-433  keep ``m`` iff ``len(m) == 2 and m[0].distance < m[1].distance * ratio``
            -> ``(m[0].trainIdx, m[0].queryIdx)``

The arithmetic lives in OpenCV's BFMatcher (third party, unpinned by the
reference; opencv-python 4.13.0 here).  Its published behaviour, restated:
distance = popcount(a XOR b) summed over the descriptor bytes; the k best train
descriptors per query in ascending distance, ties resolved toward the LOWER
train index (a stable selection); fewer than k train descriptors -> a shorter
list.  ``tests/test_oracle_match.py`` pins this restatement against
``cv2.BFMatcher(cv2.NORM_HAMMING).knnMatch`` itself, including forced ties.

Below it, the exact restatements the recalibration kernels are held to bit for bit
(``tests/test_gpu_recalib_exact.py``): the L2 matcher in float32 in the kernel's
order (``l2_top2_f32``, pinned against ``cv2.BFMatcher(cv2.NORM_L2)`` on
integer-valued descriptors), the 4-point solve of ``mcs_ransac.cu`` in float64
(``homography_4pt_exact``), its float32 inlier test (``ransac_counts_f32``) and
the Hamming launcher's queries-per-CTA choice (``match_qpc``).
"""
import math

import numpy as np

_POPCOUNT = np.array([bin(i).count("1") for i in range(256)], dtype=np.uint8)


def hamming_matrix(featuresA, featuresB):
    """All-pairs Hamming distances, int32 [len(A), len(B)]."""
    a = np.ascontiguousarray(featuresA, dtype=np.uint8)
    b = np.ascontiguousarray(featuresB, dtype=np.uint8)
    out = np.zeros((len(a), len(b)), dtype=np.int32)
    for lo in range(0, len(a), 256):   # bounded temporaries
        x = a[lo:lo + 256, None, :] ^ b[None, :, :]
        out[lo:lo + 256] = _POPCOUNT[x].sum(axis=2, dtype=np.int32)
    return out


def knn_top2(featuresA, featuresB):
    """``knnMatch(k=2)`` as arrays: ``idx`` [N,2] int32 train indices and ``dist``
    [N,2] int32 distances, best first, -1 where the train set is too small."""
    n, m = len(featuresA), len(featuresB)
    idx = -np.ones((n, 2), dtype=np.int32)
    dist = -np.ones((n, 2), dtype=np.int32)
    if n == 0 or m == 0:
        return idx, dist
    d = hamming_matrix(featuresA, featuresB)
    order = np.argsort(d, axis=1, kind="stable")[:, :2]   # stable: lower train index wins ties
    k = order.shape[1]
    idx[:, :k] = order
    dist[:, :k] = np.take_along_axis(d, order, axis=1)
    return idx, dist


def knn_top2_large(featuresA, featuresB):
    """``knn_top2`` for train sets too large for the all-pairs matrix (and for cv2's BFMatcher, which takes
    fewer than 2^18 train rows): one query at a time over 64-bit words, the best two under the order
    (distance, train index) by two first-occurrence ``argmin``s."""
    a = np.ascontiguousarray(featuresA, dtype=np.uint8)
    b = np.ascontiguousarray(featuresB, dtype=np.uint8)
    n, m = len(a), len(b)
    idx = -np.ones((n, 2), dtype=np.int32)
    dist = -np.ones((n, 2), dtype=np.int32)
    if n == 0 or m == 0:
        return idx, dist
    aw, bw = a.view(np.uint64), b.view(np.uint64)
    for i in range(n):
        d = np.bitwise_count(bw ^ aw[i]).sum(axis=1, dtype=np.int32)
        for j in range(min(2, m)):
            idx[i, j] = int(np.argmin(d))
            dist[i, j] = d[idx[i, j]]
            d[idx[i, j]] = np.iinfo(np.int32).max
    return idx, dist


def ratio_test(idx, dist, ratio=0.75):
    """The loop of StitcherClass.py:428-433.  The comparison is evaluated like the
    reference's Python expression: float distances, ``d1 * ratio`` in float64."""
    keep = np.zeros(len(idx), dtype=bool)
    matches = []
    for i in range(len(idx)):
        if idx[i, 1] >= 0 and float(dist[i, 0]) < float(dist[i, 1]) * ratio:
            keep[i] = True
            matches.append((int(idx[i, 0]), i))   # (trainIdx, queryIdx)
    return keep, matches


def match(featuresA, featuresB, ratio=0.75):
    idx, dist = knn_top2(featuresA, featuresB)
    keep, matches = ratio_test(idx, dist, ratio)
    return idx, dist, keep, matches


def match_qpc(nq_max, batch):
    """Queries per CTA the Hamming launcher of ``mcs_match.cu`` picks: start at 32 (4 per warp) and step down
    by 8 while the grid ``ceil(nq_max / qpc) x batch`` stays under two CTAs per SM of the B200 (2 x 148)."""
    qpc = 32
    while qpc > 8 and -(-nq_max // qpc) * batch < 2 * 148:
        qpc -= 8
    return qpc


# ---------------------------------------------------------------------------
# L2 (float descriptors), restated in the order mcs_match_l2_kernel evaluates it
def l2_top2_f32(featuresA, featuresB, ratio=0.75):
    """``knnMatch(k=2)`` under NORM_L2 + the ratio loop, every operation in float32 in the kernel's order:
    ``acc = 0; for k ascending: d = a_k - b_k; acc = acc + d * d``, then ``sqrt``; the two best trains per query
    under the order (distance, train index) - what cv2's ``batchDistance`` keeps, since it compares the
    square-rooted distances and inserts with a strict ``<``; the ratio rule of ``ratio_test`` in float64.

    ``featuresA`` [..., NQ, D], ``featuresB`` [..., NT, D] float32 (leading batch axes broadcast).  Returns
    ``(idx [..., NQ, 2] int32, dist [..., NQ, 2] float32, keep [..., NQ] bool)``, -1 where the train set is
    too small."""
    a = np.asarray(featuresA, dtype=np.float32)
    b = np.asarray(featuresB, dtype=np.float32)
    nt = b.shape[-2]
    lead = np.broadcast_shapes(a.shape[:-2], b.shape[:-2])
    nq = a.shape[-2]
    idx = -np.ones(lead + (nq, 2), np.int32)
    dist = -np.ones(lead + (nq, 2), np.float32)
    if nq and nt:
        acc = np.zeros(lead + (nq, nt), np.float32)
        d = np.empty_like(acc)
        for k in range(a.shape[-1]):
            np.subtract(a[..., :, None, k], b[..., None, :, k], out=d)
            np.multiply(d, d, out=d)
            np.add(acc, d, out=acc)
        dd = np.sqrt(acc)
        m = min(2, nt)
        order = np.argsort(dd, axis=-1, kind="stable")[..., :m]     # stable: the lower train index wins ties
        idx[..., :m] = order
        dist[..., :m] = np.take_along_axis(dd, order, axis=-1)
    keep = (idx[..., 1] >= 0) & (dist[..., 0].astype(np.float64) < dist[..., 1].astype(np.float64) * float(ratio))
    return idx, dist, keep


# ---------------------------------------------------------------------------
# RANSAC scoring restated op by op as mcs_ransac.cu evaluates it (float64 solve, float32 scoring)
def _square_to_quad(x, y):
    dx1, dx2, sx = x[1] - x[2], x[3] - x[2], x[0] - x[1] + x[2] - x[3]
    dy1, dy2, sy = y[1] - y[2], y[3] - y[2], y[0] - y[1] + y[2] - y[3]
    den = dx1 * dy2 - dy1 * dx2
    scale = abs(dx1) + abs(dx2) + abs(dy1) + abs(dy2)
    if not abs(den) > 1e-12 * scale * scale:
        return None
    g = (sx * dy2 - sy * dx2) / den
    h = (dx1 * sy - dy1 * sx) / den
    return [x[1] - x[0] + g * x[1], x[3] - x[0] + h * x[3], x[0],
            y[1] - y[0] + g * y[1], y[3] - y[0] + h * y[3], y[0],
            g, h, 1.0]


def homography_4pt_exact(a4, b4):
    """``homography_4pt`` of ``mcs_ransac.cu`` in Python floats (IEEE float64, no contraction: the library is
    built with ``--fmad=false``), in the kernel's order: the orientation test on the cyclic triples, the unit
    square -> quad maps of both quads, ``H = SB . adj(SA)`` summed left to right, ``H[i] *= 1 / h8``, the
    finiteness checks.  ``a4``/``b4``: the 4 x 2 float32 points of the sample.  Returns the 9 coefficients
    (float64, ``H[8] = 1``) or None where the kernel rejects the sample (count -1, ``H_k`` zero)."""
    ax, ay = [float(v) for v in np.asarray(a4)[:, 0]], [float(v) for v in np.asarray(a4)[:, 1]]
    bx, by = [float(v) for v in np.asarray(b4)[:, 0]], [float(v) for v in np.asarray(b4)[:, 1]]

    def cross(x, y, i, j, k):
        return (x[j] - x[i]) * (y[k] - y[i]) - (y[j] - y[i]) * (x[k] - x[i])

    for i in range(4):
        j, k = (i + 1) & 3, (i + 2) & 3
        if not cross(ax, ay, i, j, k) * cross(bx, by, i, j, k) > 0.0:
            return None
    SA, SB = _square_to_quad(ax, ay), _square_to_quad(bx, by)
    if SA is None or SB is None:
        return None
    adj = [SA[4] * SA[8] - SA[5] * SA[7], SA[2] * SA[7] - SA[1] * SA[8], SA[1] * SA[5] - SA[2] * SA[4],
           SA[5] * SA[6] - SA[3] * SA[8], SA[0] * SA[8] - SA[2] * SA[6], SA[2] * SA[3] - SA[0] * SA[5],
           SA[3] * SA[7] - SA[4] * SA[6], SA[1] * SA[6] - SA[0] * SA[7], SA[0] * SA[4] - SA[1] * SA[3]]
    H = [SB[3 * r] * adj[c] + SB[3 * r + 1] * adj[3 + c] + SB[3 * r + 2] * adj[6 + c]
         for r in range(3) for c in range(3)]
    h8 = H[8]
    if not abs(h8) > 1e-300 or not math.isfinite(h8):
        return None
    inv = 1.0 / h8
    H = [v * inv for v in H]
    if not all(math.isfinite(v) for v in H):
        return None
    H[8] = 1.0
    return np.array(H, dtype=np.float64)


def ransac_counts_f32(H, a, b, thresh):
    """OpenCV's ``computeError`` as ``is_inlier`` of ``mcs_ransac.cu`` evaluates it, in float32:
    ``Hf = float32(H)``, ``ww = 1 / ((Hf6 ax + Hf7 ay) + 1)``, ``dx = ((Hf0 ax + Hf1 ay) + Hf2) ww - bx`` (``dy``
    likewise), inlier iff ``dx dx + dy dy <= float32(thresh) * float32(thresh)``.  ``H``: 9 coefficients;
    ``a``/``b``: N x 2 float32.  Returns ``(count, mask N bool)``."""
    f = np.float32
    Hf = np.asarray(H, dtype=np.float64).reshape(9).astype(f)
    a = np.asarray(a, dtype=f).reshape(-1, 2)
    b = np.asarray(b, dtype=f).reshape(-1, 2)
    ax, ay, bx, by = a[:, 0], a[:, 1], b[:, 0], b[:, 1]
    with np.errstate(all="ignore"):
        ww = f(1) / (Hf[6] * ax + Hf[7] * ay + f(1))
        dx = (Hf[0] * ax + Hf[1] * ay + Hf[2]) * ww - bx
        dy = (Hf[3] * ax + Hf[4] * ay + Hf[5]) * ww - by
        mask = dx * dx + dy * dy <= f(thresh) * f(thresh)
    return int(mask.sum()), mask


# ---------------------------------------------------------------------------
# RANSAC scoring, restated for the per-hypothesis outputs of mcs_ransac_homography
def homography_from_4(a, b):
    """Exact homography through 4 correspondences a -> b (float64, h22 = 1):
    the 8x8 linear system of the minimal solver OpenCV's RANSAC runs per sample
    (cv::findHomography -> HomographyEstimatorCallback::runKernel on 4 points).
    Returns None for a singular system."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    A = np.zeros((8, 8))
    rhs = np.zeros(8)
    for i in range(4):
        x, y = a[i]
        u, v = b[i]
        A[2 * i] = [x, y, 1, 0, 0, 0, -u * x, -u * y]
        A[2 * i + 1] = [0, 0, 0, x, y, 1, -v * x, -v * y]
        rhs[2 * i] = u
        rhs[2 * i + 1] = v
    try:
        h = np.linalg.solve(A, rhs)
    except np.linalg.LinAlgError:
        return None
    if not np.all(np.isfinite(h)):
        return None
    return np.append(h, 1.0).reshape(3, 3)


def sample_is_valid(a, b):
    """The sample filter of cv::findHomography's RANSAC (HomographyEstimatorCallback::
    checkSubset): for every cyclic triple of the 4 correspondences the orientation
    (sign of the cross product) must be the same, and non-zero, in both images."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)

    def cross(p, i, j, k):
        return (p[j, 0] - p[i, 0]) * (p[k, 1] - p[i, 1]) - (p[j, 1] - p[i, 1]) * (p[k, 0] - p[i, 0])

    for i in range(4):
        j, k = (i + 1) % 4, (i + 2) % 4
        if not cross(a, i, j, k) * cross(b, i, j, k) > 0.0:
            return False
    return True


def reprojection_errors_sq(H, a, b):
    """Squared forward reprojection error of every correspondence (the inlier
    criterion of cv::findHomography's RANSAC: err <= thresh^2)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    w = H[2, 0] * a[:, 0] + H[2, 1] * a[:, 1] + H[2, 2]
    x = (H[0, 0] * a[:, 0] + H[0, 1] * a[:, 1] + H[0, 2]) / w
    y = (H[1, 0] * a[:, 0] + H[1, 1] * a[:, 1] + H[1, 2]) / w
    return (x - b[:, 0]) ** 2 + (y - b[:, 1]) ** 2


def corner_error(H1, H2, w, h):
    """Max distance between the images of the frame corners under two homographies."""
    c = np.array([[0, 0, 1], [w, 0, 1], [w, h, 1], [0, h, 1]], dtype=np.float64).T
    p1 = H1 @ c
    p2 = H2 @ c
    p1 = p1[:2] / p1[2]
    p2 = p2[:2] / p2[2]
    return float(np.sqrt(((p1 - p2) ** 2).sum(axis=0)).max())
