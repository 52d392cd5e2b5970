"""ORACLE (test infrastructure, never imported by the product package).

Exposure compensation of the camera-weighted and multi-band blends (include/mcs.h mcs_plan_estimate_gains,
mcs_plan_set_exposure_gains): OpenCV's ``cv::detail::GainCompensator``, the class
``cv2.detail.ExposureCompensator_createDefault(GAIN)`` returns, run on the planes of ``multiband_model.camera_planes``
- the layers with a non-empty clipped rectangle, innermost first - with ``corners[k]`` the rectangle's ``(x0, y0)``,
``images[k]`` the 3-channel overwrite sample ``v_k`` and ``masks[k]`` the weight sample ``w_k`` itself (255 without a
map): the uncut weights, the same masks the seam finders get, so seams do not change the gains.

``gains_cv2`` - the definition: ``feed(corners, images, masks)`` and ``getMatGains()``.

``stats`` - its statistics, exactly: for every pair ``i <= j`` in feed order whose rectangles overlap
(``seam_model.overlap``; ``i == j`` included), ``intersect = (m_i == 255) & (m_j == 255)`` over the overlap - only the
value 255 counts, so ramps below 255 and the bilinear rim of a warped camera, which the zero border darkens, drop out
by construction - ``N(i, j) = N(j, i) = max(1, count)``, and for ``i != j``
``I(i, j) = Isum_i / N(i, j)``, ``I(j, i) = Isum_j / N(i, j)``, where ``Isum_c`` is the sequential float64 sum, in
row-major order over the overlap, of ``sqrt(double(b^2 + g^2 + r^2))`` of camera c's intersect pixels.  ``N`` is 0
for rectangles that do not overlap; ``I(i, i)`` is never used and stays 0.  ``skip[i]`` marks a camera that shares
no intersect pixel with any other camera.

``solve`` - the gains from the statistics: with ``alpha = 0.01``, ``beta = 100`` and ``k`` running over the cameras
not skipped, ``b(ki) += beta N(i, j)`` and ``A(ki, ki) += beta N(i, j)`` over every such j (i included), and for
``j != i`` ``A(ki, ki) += 2 alpha I(i, j)^2 N(i, j)``, ``A(ki, kj) -= 2 alpha I(i, j) I(j, i) N(i, j)``, each in that
order and association; then ``A g = b`` by Gaussian elimination with partial pivoting (the ``LUImpl`` of OpenCV's
``hal::LU64f``: ``d = -1 / pivot``, row updates ``A[j][k] += (A[j][i] d) A[i][k]``, back substitution
``(b_i - sum A[i][k] g_k) / A[i][i]``) in plain float64 without contraction.  Skipped cameras keep gain 1.  ``A`` is
symmetric positive definite (its diagonal holds ``beta N(i, i) >= 100``), so no pivot vanishes.  ``cv2.solve`` runs the
same elimination through a SIMD inner loop whose rounding depends on the build (and Cramer's rule for 3 unknowns):
from 3 unknowns on the two differ in the last bits, which the CPU tests bound.

``lut(g)`` - what ``apply`` does to every sample value: ``saturate_u8(rint_half_even(v * g))`` in float64, one gain
on every channel (alpha included); ``apply`` / ``apply_cv2`` on images of 1, 3 or 4 channels.  They agree while
``255 g < 2^31``; beyond, cv2's conversion to int overflows, and the table saturates to 255.

``blend_weighted`` / ``blend_multiband`` - ``camera_weight_model`` / ``multiband_model`` with every camera's
sample ``v_k`` replaced by ``lut_k[v_k]`` (with Voronoi seams or graph-cut seams, the latter found on the
compensated samples of ``seam_frames``); their ``_cv2`` forms estimate with ``gains_cv2``, compensate with the cv2
class's ``apply`` and blend with ``combine`` / ``blend_planes_cv2``.  ``gains`` are indexed by ``layer.cam`` like
``frames`` and ``maps``; None estimates them on ``frames``.
"""
import numpy as np

from . import camera_weight_model as cw
from . import multiband_model as mb
from .graphcut_seam_model import plane_inputs
from .seam_model import overlap

ALPHA = 0.01
BETA = 100.0


def _crop(a, corner, roi):
    rx0, ry0, rx1, ry1 = roi
    return a[ry0 - corner[1]:ry1 - corner[1], rx0 - corner[0]:rx1 - corner[0]]


def norms(image):
    """``cv::norm`` of every 3-channel u8 pixel: ``sqrt(double(b^2 + g^2 + r^2))`` (the squares are exact)."""
    v = np.asarray(image).astype(np.int64)
    return np.sqrt((v * v).sum(axis=2).astype(np.float64))


def seq_sum(values):
    """The sequential float64 sum ``((v_0 + v_1) + v_2) + ...`` (``np.cumsum`` adds left to right; ``np.sum`` would
    add pairwise)."""
    values = np.asarray(values, np.float64)
    return float(np.cumsum(values)[-1]) if values.size else 0.0


def stats(sizes, corners, masks, images):
    """``(N, I, skip)``: int64 n x n, float64 n x n, bool n.  ``images[k]``: h x w x 3 uint8 of plane k."""
    n = len(masks)
    N = np.zeros((n, n), np.int64)
    I = np.zeros((n, n), np.float64)
    skip = np.ones(n, bool)
    for i in range(n):
        for j in range(i, n):
            roi = overlap(sizes[i], corners[i], sizes[j], corners[j])
            if roi is None:
                continue
            inter = (_crop(np.asarray(masks[i]), corners[i], roi) == 255) & (_crop(np.asarray(masks[j]), corners[j], roi) == 255)
            count = int(inter.sum())
            N[i, j] = N[j, i] = max(1, count)
            if count == 0 or i == j:
                continue
            skip[i] = skip[j] = False
            I[i, j] = seq_sum(norms(_crop(images[i], corners[i], roi))[inter]) / N[i, j]
            I[j, i] = seq_sum(norms(_crop(images[j], corners[j], roi))[inter]) / N[i, j]
    return N, I, skip


def normal_equations(N, I, skip):
    """``(A, b, cams)`` of the cameras not skipped (lists of Python floats), in OpenCV's order of additions."""
    cams = [i for i in range(len(skip)) if not skip[i]]
    m = len(cams)
    A = [[0.0] * m for _ in range(m)]
    b = [0.0] * m
    for ki, i in enumerate(cams):
        for kj, j in enumerate(cams):
            nij, iij, iji = float(N[i, j]), float(I[i, j]), float(I[j, i])
            b[ki] += BETA * nij
            A[ki][ki] += BETA * nij
            if j != i:
                A[ki][ki] += 2 * ALPHA * iij * iij * nij
                A[ki][kj] -= 2 * ALPHA * iij * iji * nij
    return A, b, cams


def lu_solve(A, b):
    """OpenCV's ``LUImpl`` on copies of ``A`` (m x m) and ``b`` (m), operation for operation."""
    A = [list(map(float, r)) for r in A]
    b = [float(v) for v in b]
    m = len(b)
    for i in range(m):
        k = i
        for j in range(i + 1, m):
            if abs(A[j][i]) > abs(A[k][i]):
                k = j
        if k != i:
            A[i][i:], A[k][i:] = A[k][i:], A[i][i:]
            b[i], b[k] = b[k], b[i]
        d = -1.0 / A[i][i]
        for j in range(i + 1, m):
            alpha = A[j][i] * d
            for c in range(i + 1, m):
                A[j][c] += alpha * A[i][c]
            b[j] += alpha * b[i]
    for i in range(m - 1, -1, -1):
        s = b[i]
        for c in range(i + 1, m):
            s -= A[i][c] * b[c]
        b[i] = s / A[i][i]
    return b


def solve(N, I, skip):
    """The gains (float64 n) from the statistics, by ``lu_solve``."""
    A, b, cams = normal_equations(N, I, skip)
    out = np.ones(len(skip), np.float64)
    for k, g in zip(cams, lu_solve(A, b)):
        out[k] = g
    return out


def solve_cv2(N, I, skip):
    """The same normal equations through ``cv2.solve`` (what ``GainCompensator`` calls)."""
    import cv2
    A, b, cams = normal_equations(N, I, skip)
    out = np.ones(len(skip), np.float64)
    if cams:
        ok, g = cv2.solve(np.array(A, np.float64), np.array(b, np.float64).reshape(-1, 1))
        assert ok
        out[cams] = g.ravel()
    return out


def gains(sizes, corners, masks, images):
    """``solve(*stats(...))``."""
    return solve(*stats(sizes, corners, masks, images))


def gains_cv2(sizes, corners, masks, images):
    """The definition: ``GainCompensator.feed`` and ``getMatGains``."""
    import cv2
    cv2.ocl.setUseOpenCL(False)
    comp = cv2.detail.ExposureCompensator_createDefault(cv2.detail.ExposureCompensator_GAIN)
    comp.feed(corners=[(int(x), int(y)) for x, y in corners],
              images=[np.ascontiguousarray(v, np.uint8) for v in images],
              masks=[np.ascontiguousarray(m, np.uint8) for m in masks])
    return np.array([float(np.asarray(g).ravel()[0]) for g in comp.getMatGains()], np.float64)


def lut(g):
    """The 256-entry u8 table of gain ``g``: ``saturate_u8(rint_half_even(v * g))``."""
    return np.clip(np.rint(np.arange(256, dtype=np.float64) * float(g)), 0, 255).astype(np.uint8)


def apply(image, g):
    return lut(g)[np.asarray(image, np.uint8)]


def apply_cv2(image, g):
    """``GainCompensator.apply`` with the gain set to ``g`` (on a copy: cv2 compensates in place)."""
    import cv2
    comp = cv2.detail.ExposureCompensator_createDefault(cv2.detail.ExposureCompensator_GAIN)
    comp.setMatGains([np.array([[float(g)]], np.float64)])
    img = np.array(image, np.uint8, copy=True)
    return comp.apply(0, (0, 0), img, np.full(img.shape[:2], 255, np.uint8))


# ---- the blends ---------------------------------------------------------------------------------------------------
def fed_cams(layers, out_w, out_h):
    """``layer.cam`` of the layers with a non-empty clipped rectangle, in feed order (the order of ``camera_planes``)."""
    out = []
    for l in layers:
        x0, y0, x1, y1 = [int(v) for v in l.rect]
        if min(out_w, x1) > max(0, x0) and min(out_h, y1) > max(0, y0):
            out.append(l.cam)
    return out


def camera_gains(layers, out_w, out_h, frames, maps, estimator=gains):
    """Per camera (indexed by ``layer.cam``), the gains estimated on the samples of 3-channel ``frames``; 1 for a
    camera whose layer feeds nothing."""
    planes = mb.camera_planes(layers, out_w, out_h, frames, maps)
    out = [1.0] * (max(l.cam for l in layers) + 1)
    if planes:
        for cam, g in zip(fed_cams(layers, out_w, out_h), estimator(*plane_inputs(planes))):
            out[cam] = float(g)
    return out


def compensated_planes(layers, out_w, out_h, frames, maps, gains, use_cv2=False):
    """``multiband_model.camera_planes`` with every ``v_k`` replaced by ``lut_k[v_k]`` (or the cv2 class's apply)."""
    planes = mb.camera_planes(layers, out_w, out_h, frames, maps)
    comp = apply_cv2 if use_cv2 else apply
    return [(r, comp(v, gains[cam]), w) for (r, v, w), cam in zip(planes, fed_cams(layers, out_w, out_h))]


def _as_out(out, frames, layers):
    return out[:, :, 0] if np.asarray(frames[layers[0].cam]).ndim == 2 else out


def _weighted(layers, out_w, out_h, frames, maps, gains, use_cv2):
    C = mb._as3(frames[layers[0].cam]).shape[2]
    values, weights, reaches = [], [], []
    for (x0, y0, x1, y1), v, w in compensated_planes(layers, out_w, out_h, frames, maps, gains, use_cv2):
        V = np.zeros((out_h, out_w, C), np.uint8)
        Wt = np.zeros((out_h, out_w), np.int64)
        R = np.zeros((out_h, out_w), bool)
        V[y0:y1, x0:x1], Wt[y0:y1, x0:x1], R[y0:y1, x0:x1] = v, w, True
        values.append(V)
        weights.append(Wt)
        reaches.append(R)
    if not values:
        return _as_out(np.zeros((out_h, out_w, C), np.uint8), frames, layers)
    return _as_out(cw.combine(values, weights, reaches)[0], frames, layers)


def blend_weighted(layers, out_w, out_h, frames, maps, gains=None):
    """The camera-weighted blend (``camera_weight_model``) of the compensated samples."""
    if gains is None:
        gains = camera_gains(layers, out_w, out_h, frames, maps)
    return _weighted(layers, out_w, out_h, frames, maps, gains, False)


def blend_weighted_cv2(layers, out_w, out_h, frames, maps, gains=None):
    """The same with cv2's estimate and apply."""
    if gains is None:
        gains = camera_gains(layers, out_w, out_h, frames, maps, gains_cv2)
    return _weighted(layers, out_w, out_h, frames, maps, gains, True)


def _multiband(layers, out_w, out_h, frames, maps, bands, gains, seams, seam_frames, use_cv2):
    from . import graphcut_seam_model as gc
    from . import seam_model
    planes = compensated_planes(layers, out_w, out_h, frames, maps, gains, use_cv2)
    if planes and seams == "voronoi":
        planes = seam_model.cut_planes(planes, seam_model.find_cv2 if use_cv2 else seam_model.find)
    elif planes and seams == "graphcut":
        seam = planes if seam_frames is None else compensated_planes(layers, out_w, out_h, seam_frames, maps, gains,
                                                                     use_cv2)
        finder = gc.find_graphcut_cv2 if use_cv2 else gc.find_graphcut
        cut = finder(*gc.plane_inputs(seam))
        planes = [(r, v, c.astype(np.int64)) for (r, v, _), c in zip(planes, cut)]
    else:
        assert seams is None, seams
    C = mb._as3(frames[layers[0].cam]).shape[2]
    if use_cv2:
        return _as_out(mb.blend_planes_cv2(planes, out_w, out_h, bands, C), frames, layers)
    return _as_out(mb.blend_planes(planes, out_w, out_h, bands, C)[0], frames, layers)


def blend_multiband(layers, out_w, out_h, frames, maps, bands, gains=None, seams=None, seam_frames=None):
    """The multi-band blend (``multiband_model.blend_planes``) of the compensated samples, on the weights cut by
    ``seams`` = None, "voronoi" or "graphcut" (found on the compensated samples of ``seam_frames``, default
    ``frames``)."""
    if gains is None:
        gains = camera_gains(layers, out_w, out_h, frames, maps)
    return _multiband(layers, out_w, out_h, frames, maps, bands, gains, seams, seam_frames, False)


def blend_multiband_cv2(layers, out_w, out_h, frames, maps, bands, gains=None, seams=None, seam_frames=None):
    """The definition: cv2's compensator, seam finder and ``MultiBandBlender``."""
    if gains is None:
        gains = camera_gains(layers, out_w, out_h, frames, maps, gains_cv2)
    return _multiband(layers, out_w, out_h, frames, maps, bands, gains, seams, seam_frames, True)
