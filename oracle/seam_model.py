"""ORACLE (test infrastructure, never imported by the product package).

Voronoi seam masks for the multi-band blend (include/mcs.h mcs_plan_set_voronoi_seams): OpenCV's
``cv::detail::VoronoiSeamFinder`` run on the planes of ``multiband_model.camera_planes`` - the layers with a
non-empty clipped rectangle, innermost first.  ``sizes[k]`` is the rectangle's ``(w, h)``, ``corners[k]`` its
``(x0, y0)`` and ``masks[k]`` the uint8 weight sample ``w_k`` itself (255 without a map).  The finder only
zeroes pixels and only asks whether a mask is non-zero, so its output is the seam-cut weights: each camera's
weights survive inside its seam cell and are 0 elsewhere.

``find_cv2`` - the definition, calling the cv2 class (``createDefault``; constructing
``cv2.detail_VoronoiSeamFinder`` directly and calling ``find`` crashes in cv2 4.13).

``find`` - the same in numpy integers, as the kernels of csrc/mcs_seams.cu follow it:
  - the pairs ``(i, j)``, ``i < j``, in feed order, each pair whose rectangles overlap (``overlapRoi``); each
    pair updates the masks in place, so later pairs see what earlier pairs cut;
  - the submask is the overlap ROI grown by ``GAP`` on every side, reading 0 outside each mask;
  - ``collision = (s1 != 0) & (s2 != 0)``, ``u1 = (s1 != 0) & ~collision``, ``u2`` likewise;
  - ``d(u)`` is the exact L1 distance to the nearest pixel of ``u`` (``distanceTransform(u == 0, DIST_L1, 3)``,
    a 3 x 3 chamfer with costs 1 and 2); for an empty ``u`` it is ``EMPTY + min(y + 1, x + 1, H - y, W - x)``
    (OpenCV's INT_MAX border after the float conversion), H x W the submask's size;
  - inside the ROI, where ``d(u1) < d(u2)`` the pixel is zeroed in mask j, otherwise in mask i (ties go to the
    later camera).
Every real distance is below ``W + H``; plans with a submask of ``W + H >= EMPTY`` are refused (below that
bound every distance and the empty rule's values fit in uint16).

``blend`` / ``blend_cv2`` are ``multiband_model.blend`` / ``blend_cv2`` with every plane's ``w`` first replaced by the
seam-cut weights of ``find`` / ``find_cv2``: the panorama of the multi-band blend with Voronoi seams.
"""
import numpy as np

GAP = 10
EMPTY = 32768


def overlap(size_i, corner_i, size_j, corner_j):
    """``overlapRoi``: the intersection ``(x0, y0, x1, y1)`` of two rectangles, or None when it is empty."""
    (w1, h1), (x1, y1) = size_i, corner_i
    (w2, h2), (x2, y2) = size_j, corner_j
    rx0, ry0 = max(x1, x2), max(y1, y2)
    rx1, ry1 = min(x1 + w1, x2 + w2), min(y1 + h1, y2 + h2)
    if rx0 >= rx1 or ry0 >= ry1:
        return None
    return rx0, ry0, rx1, ry1


def submask_size(roi):
    """``(W, H)`` of the submask of an overlap ROI."""
    rx0, ry0, rx1, ry1 = roi
    return rx1 - rx0 + 2 * GAP, ry1 - ry0 + 2 * GAP


def supported(sizes, corners):
    """Whether every overlapping pair's submask keeps ``W + H`` below ``EMPTY``."""
    n = len(sizes)
    for i in range(n - 1):
        for j in range(i + 1, n):
            roi = overlap(sizes[i], corners[i], sizes[j], corners[j])
            if roi is not None and sum(submask_size(roi)) >= EMPTY:
                return False
    return True


def l1_distance(u):
    """Exact L1 distance of every pixel to the nearest pixel of the boolean plane ``u`` (int64), with the
    empty-plane rule.  Separable: the 1-D distance along each row, then ``min(h, prev + 1)`` down and up."""
    H, W = u.shape
    if not u.any():
        yy, xx = np.mgrid[0:H, 0:W]
        return EMPTY + np.minimum.reduce([yy + 1, xx + 1, H - yy, W - xx]).astype(np.int64)
    inf = 1 << 40
    x = np.arange(W, dtype=np.int64)
    left = np.maximum.accumulate(np.where(u, x[None, :], -inf), axis=1)
    right = np.minimum.accumulate(np.where(u, x[None, :], inf)[:, ::-1], axis=1)[:, ::-1]
    d = np.minimum(x[None, :] - left, right - x[None, :])
    for y in range(1, H):
        d[y] = np.minimum(d[y], d[y - 1] + 1)
    for y in range(H - 2, -1, -1):
        d[y] = np.minimum(d[y], d[y + 1] + 1)
    return d


def _sub(m, corner, roi):
    """The submask of one mask: the ROI grown by GAP, 0 outside the mask."""
    rx0, ry0, rx1, ry1 = roi
    W, H = submask_size(roi)
    s = np.zeros((H, W), np.uint8)
    ys = np.arange(H) + ry0 - GAP - corner[1]
    xs = np.arange(W) + rx0 - GAP - corner[0]
    vy = (ys >= 0) & (ys < m.shape[0])
    vx = (xs >= 0) & (xs < m.shape[1])
    s[np.ix_(vy, vx)] = m[np.ix_(ys[vy], xs[vx])]
    return s


def find(sizes, corners, masks, details=False):
    """The numpy restatement: the seam-cut masks (copies), or ``(masks, pairs)`` with ``details`` where
    ``pairs`` lists ``(i, j, roi)`` in the order they were visited."""
    masks = [np.array(m, np.uint8, copy=True) for m in masks]
    if not supported(sizes, corners):
        raise ValueError("a submask of W + H >= %d: outside the uint16 distances of the specification" % EMPTY)
    pairs = []
    n = len(masks)
    for i in range(n - 1):
        for j in range(i + 1, n):
            roi = overlap(sizes[i], corners[i], sizes[j], corners[j])
            if roi is None:
                continue
            pairs.append((i, j, roi))
            s1, s2 = _sub(masks[i], corners[i], roi), _sub(masks[j], corners[j], roi)
            collision = (s1 != 0) & (s2 != 0)
            u1 = (s1 != 0) & ~collision
            u2 = (s2 != 0) & ~collision
            first = (l1_distance(u1) < l1_distance(u2))[GAP:-GAP, GAP:-GAP]
            rx0, ry0, rx1, ry1 = roi
            m1 = masks[i][ry0 - corners[i][1]:ry1 - corners[i][1], rx0 - corners[i][0]:rx1 - corners[i][0]]
            m2 = masks[j][ry0 - corners[j][1]:ry1 - corners[j][1], rx0 - corners[j][0]:rx1 - corners[j][0]]
            m2[first] = 0
            m1[~first] = 0
    return (masks, pairs) if details else masks


def find_cv2(sizes, corners, masks):
    """The definition: ``cv2.detail.SeamFinder_createDefault(VORONOI_SEAM).find`` on the masks (copies)."""
    import cv2
    finder = cv2.detail.SeamFinder_createDefault(cv2.detail.SeamFinder_VORONOI_SEAM)
    imgs = [cv2.UMat(np.zeros((int(h), int(w), 3), np.float32)) for (w, h) in sizes]
    out = finder.find(imgs, [(int(x), int(y)) for x, y in corners],
                      [cv2.UMat(np.ascontiguousarray(m, np.uint8)) for m in masks])
    return [u.get() for u in out]


def plane_inputs(planes):
    """``(sizes, corners, masks)`` of ``multiband_model`` planes ``[(rect, v, w)]``."""
    sizes = [(x1 - x0, y1 - y0) for (x0, y0, x1, y1), _, _ in planes]
    corners = [(x0, y0) for (x0, y0, _, _), _, _ in planes]
    masks = [np.asarray(w).astype(np.uint8) for _, _, w in planes]
    return sizes, corners, masks


def cut_planes(planes, finder=find):
    """The planes with every ``w`` replaced by its seam-cut weights."""
    if not planes:
        return planes
    cut = finder(*plane_inputs(planes))
    return [(r, v, c.astype(np.int64)) for (r, v, _), c in zip(planes, cut)]


def _as_out(out, frames, layers):
    return out[:, :, 0] if np.asarray(frames[layers[0].cam]).ndim == 2 else out


def blend(layers, out_w, out_h, frames, maps, bands):
    """``multiband_model.blend`` on the weights cut by ``find``.  ``frames`` and ``maps`` are indexed by
    ``layer.cam`` (``maps[cam]`` None = 255 everywhere); the panorama is 2-D for 2-D frames."""
    from . import multiband_model as mb
    planes = cut_planes(mb.camera_planes(layers, out_w, out_h, frames, maps), find)
    C = mb._as3(frames[layers[0].cam]).shape[2]
    return _as_out(mb.blend_planes(planes, out_w, out_h, bands, C)[0], frames, layers)


def blend_cv2(layers, out_w, out_h, frames, maps, bands):
    """The definition: ``cv2.detail_MultiBandBlender`` (``multiband_model.blend_planes_cv2``) on the weights cut by
    cv2's VoronoiSeamFinder."""
    from . import multiband_model as mb
    planes = cut_planes(mb.camera_planes(layers, out_w, out_h, frames, maps), find_cv2)
    C = mb._as3(frames[layers[0].cam]).shape[2]
    return _as_out(mb.blend_planes_cv2(planes, out_w, out_h, bands, C), frames, layers)
