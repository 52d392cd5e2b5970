"""ORACLE (test infrastructure, never imported by the product package).

Graph-cut seam masks for the multi-band blend (include/mcs.h mcs_plan_set_graphcut_seams): OpenCV's
``cv::detail::GraphCutSeamFinder("COST_COLOR")`` run on the planes of ``multiband_model.camera_planes`` - the layers
with a non-empty clipped rectangle, innermost first - with ``sizes[k]`` the rectangle's ``(w, h)``, ``corners[k]`` its
``(x0, y0)``, ``masks[k]`` the uint8 weight sample ``w_k`` (255 without a map) and ``images[k]`` the 3-channel
overwrite sample ``v_k`` of one frame-set.  Like ``seam_model``'s Voronoi finder it only zeroes mask pixels, so its
output is the cut weights.

``find_graphcut_cv2`` - the definition, calling the cv2 class on ``CV_32FC3`` images.

``find_graphcut`` - the same with exact integers, as csrc/mcs_seams_graphcut.cu follows it:
  - the pairs ``(i, j)``, ``i < j``, in feed order, each pair whose rectangles overlap (``seam_model.overlap``); each
    pair updates the masks in place, so later pairs cut what earlier pairs left;
  - the submask is the overlap ROI grown by ``GAP`` on every side, masks and images reading 0 outside each plane;
  - ``D(p) = sum_c (I1_c(p) - I2_c(p))^2`` on the two image submasks;
  - terminal edges: ``TERMINAL`` from the source where ``s1 != 0``, ``TERMINAL`` to the sink where ``s2 != 0``
    (a pixel with both is the same as one with neither, up to a constant, and is built as one with neither);
  - each 4-neighbour pair ``p, q`` gets ``D(p) + D(q) + 1`` in both directions, plus ``PENALTY`` when any of
    ``s1(p), s1(q), s2(p), s2(q)`` is 0;
  - the cut is ``S``, the pixels reachable from the source in the residual graph of a maximum flow: the minimal
    source side of a minimum cut, the same for every maximum flow;
  - inside the ROI, ``p`` in ``S`` with ``s1(p) != 0`` is zeroed in mask j, ``p`` not in ``S`` with ``s2(p) != 0`` in
    mask i.
Every capacity is an integer below 2^21 (cv2's float graph computes the same flows exactly).  Where several cuts
cost the minimum - flat or identical content, ``D = 0`` - cv2 returns whichever its Boykov-Kolmogorov search order
finds; ``find_graphcut`` returns the minimal source side, a rule with no hidden state.  On textured content the two
agree on every pixel.  The max flow is scipy's (seconds for ~10^5-pixel submasks): an oracle for small rigs.

``blend_graphcut`` / ``blend_graphcut_cv2`` are the multi-band blend of ``frames`` (``multiband_model.blend_planes`` /
``blend_planes_cv2``) on the weights cut by ``find_graphcut`` / ``find_graphcut_cv2`` on the samples of
``seam_frames`` (default: ``frames``).
"""
import numpy as np

from .seam_model import overlap

GAP = 10           # the overlap ROI grows by this much on every side (as for the Voronoi finder)
TERMINAL = 10000   # GraphCutSeamFinder's terminal_cost
PENALTY = 1000     # its bad_region_penalty


def submask_size(roi):
    """``(W, H)`` of the submask of an overlap ROI."""
    rx0, ry0, rx1, ry1 = roi
    return rx1 - rx0 + 2 * GAP, ry1 - ry0 + 2 * GAP


def sub(a, corner, roi):
    """The submask of one plane (H x W or H x W x C): the ROI grown by GAP, 0 outside the plane."""
    rx0, ry0, rx1, ry1 = roi
    W, H = submask_size(roi)
    s = np.zeros((H, W) + a.shape[2:], a.dtype)
    ys = np.arange(H) + ry0 - GAP - corner[1]
    xs = np.arange(W) + rx0 - GAP - corner[0]
    vy = (ys >= 0) & (ys < a.shape[0])
    vx = (xs >= 0) & (xs < a.shape[1])
    s[np.ix_(vy, vx)] = a[np.ix_(ys[vy], xs[vx])]
    return s


def graphcut_graph(s1, s2, i1, i2, pin_source=None, pin_sink=None):
    """The flow network of one pair's submasks: ``(csr capacities, source, sink, n)`` with pixel ``y * W + x`` as
    node ``y * W + x``, the source ``n`` and the sink ``n + 1``.  ``pin_source`` / ``pin_sink`` (boolean H x W) add
    terminal edges of 2^30 - more than every real cut - to force pixels onto one side."""
    import scipy.sparse as sp
    H, W = s1.shape
    n = H * W
    a1, a2 = s1.ravel() != 0, s2.ravel() != 0
    d = ((i1.astype(np.int64) - i2.astype(np.int64)) ** 2).sum(axis=2)
    ok = (s1 != 0) & (s2 != 0)
    idx = np.arange(n).reshape(H, W)
    rows, cols, caps = [], [], []
    src = np.where(a1 & ~a2, TERMINAL, 0)
    snk = np.where(a2 & ~a1, TERMINAL, 0)
    if pin_source is not None:
        src = src + np.where(pin_source.ravel(), 1 << 30, 0)
    if pin_sink is not None:
        snk = snk + np.where(pin_sink.ravel(), 1 << 30, 0)
    for cap, to_sink in ((src, False), (snk, True)):
        nz = np.nonzero(cap)[0]
        rows.append(nz if to_sink else np.full(nz.size, n))
        cols.append(np.full(nz.size, n + 1) if to_sink else nz)
        caps.append(cap[nz])
    wh = d[:, :-1] + d[:, 1:] + 1 + np.where(ok[:, :-1] & ok[:, 1:], 0, PENALTY)
    wv = d[:-1, :] + d[1:, :] + 1 + np.where(ok[:-1, :] & ok[1:, :], 0, PENALTY)
    for w, p, q in ((wh, idx[:, :-1], idx[:, 1:]), (wv, idx[:-1, :], idx[1:, :])):
        rows += [p.ravel(), q.ravel()]
        cols += [q.ravel(), p.ravel()]
        caps += [w.ravel(), w.ravel()]
    caps = np.concatenate(caps)
    assert caps.max(initial=0) < 1 << 31
    M = sp.csr_matrix((caps.astype(np.int32), (np.concatenate(rows), np.concatenate(cols))), shape=(n + 2, n + 2))
    return M, n, n + 1, n


def min_cut(M, source, sink, method="dinic"):
    """``(flow value, reachable)``: a maximum flow (scipy) and the nodes reachable from ``source`` in its residual
    graph (boolean, every node)."""
    from scipy.sparse.csgraph import breadth_first_order, maximum_flow
    r = maximum_flow(M, source, sink, method=method)
    R = (M - r.flow).tocsr()
    R.data = (R.data > 0).astype(np.int8)
    R.eliminate_zeros()
    reach = np.zeros(M.shape[0], bool)
    reach[breadth_first_order(R, source, directed=True, return_predecessors=False)] = True
    assert not reach[sink]
    return int(r.flow_value), reach


def graphcut_side(s1, s2, i1, i2, method="dinic"):
    """``S`` of one pair: boolean H x W, True on the source side (camera i)."""
    M, source, sink, n = graphcut_graph(s1, s2, i1, i2)
    return min_cut(M, source, sink, method)[1][:n].reshape(s1.shape)


def find_graphcut(sizes, corners, masks, images, details=False, method="dinic"):
    """The integer restatement: the graph-cut masks (copies), or ``(masks, pairs)`` with ``details`` where ``pairs``
    lists ``(i, j, roi)`` in the order they were visited.  ``images[k]``: h x w x 3 of plane k."""
    masks = [np.array(m, np.uint8, copy=True) for m in masks]
    images = [np.asarray(v) for v in images]
    pairs = []
    n = len(masks)
    for i in range(n - 1):
        for j in range(i + 1, n):
            roi = overlap(sizes[i], corners[i], sizes[j], corners[j])
            if roi is None:
                continue
            pairs.append((i, j, roi))
            s1, s2 = sub(masks[i], corners[i], roi), sub(masks[j], corners[j], roi)
            i1, i2 = sub(images[i], corners[i], roi), sub(images[j], corners[j], roi)
            side = graphcut_side(s1, s2, i1, i2, method)[GAP:-GAP, GAP:-GAP]
            in1, in2 = (s1 != 0)[GAP:-GAP, GAP:-GAP], (s2 != 0)[GAP:-GAP, GAP:-GAP]
            rx0, ry0, rx1, ry1 = roi
            m1 = masks[i][ry0 - corners[i][1]:ry1 - corners[i][1], rx0 - corners[i][0]:rx1 - corners[i][0]]
            m2 = masks[j][ry0 - corners[j][1]:ry1 - corners[j][1], rx0 - corners[j][0]:rx1 - corners[j][0]]
            m2[side & in1] = 0
            m1[~side & in2] = 0
    return (masks, pairs) if details else masks


def find_graphcut_cv2(sizes, corners, masks, images):
    """The definition: ``cv2.detail_GraphCutSeamFinder("COST_COLOR").find`` on ``CV_32FC3`` images (copies)."""
    import cv2
    finder = cv2.detail_GraphCutSeamFinder("COST_COLOR")
    imgs = [cv2.UMat(np.ascontiguousarray(v, np.float32)) for v in images]
    out = finder.find(imgs, [(int(x), int(y)) for x, y in corners],
                      [cv2.UMat(np.ascontiguousarray(m, np.uint8)) for m in masks])
    return [u.get() for u in out]


def plane_inputs(planes):
    """``(sizes, corners, masks, images)`` of ``multiband_model`` planes ``[(rect, v, w)]``: the samples ``v`` as
    uint8 h x w x C."""
    sizes = [(x1 - x0, y1 - y0) for (x0, y0, x1, y1), _, _ in planes]
    corners = [(x0, y0) for (x0, y0, _, _), _, _ in planes]
    masks = [np.asarray(w).astype(np.uint8) for _, _, w in planes]
    images = [np.asarray(v).astype(np.uint8) for _, v, _ in planes]
    return sizes, corners, masks, images


def graphcut_planes(layers, out_w, out_h, frames, maps, seam_frames=None, finder=find_graphcut):
    """The planes of ``frames`` with every ``w`` replaced by its graph-cut weights, found on the samples of
    ``seam_frames`` (default ``frames``; 3-channel)."""
    from . import multiband_model as mb
    planes = mb.camera_planes(layers, out_w, out_h, frames, maps)
    if not planes:
        return planes
    seam = planes if seam_frames is None else mb.camera_planes(layers, out_w, out_h, seam_frames, maps)
    cut = finder(*plane_inputs(seam))
    return [(r, v, c.astype(np.int64)) for (r, v, _), c in zip(planes, cut)]


def _as_out(out, frames, layers):
    return out[:, :, 0] if np.asarray(frames[layers[0].cam]).ndim == 2 else out


def blend_graphcut(layers, out_w, out_h, frames, maps, bands, seam_frames=None):
    """``multiband_model.blend`` on the weights cut by ``find_graphcut`` on ``seam_frames`` (default ``frames``)."""
    from . import multiband_model as mb
    planes = graphcut_planes(layers, out_w, out_h, frames, maps, seam_frames)
    C = mb._as3(frames[layers[0].cam]).shape[2]
    return _as_out(mb.blend_planes(planes, out_w, out_h, bands, C)[0], frames, layers)


def blend_graphcut_cv2(layers, out_w, out_h, frames, maps, bands, seam_frames=None):
    """The definition: ``cv2.detail_MultiBandBlender`` on the weights cut by cv2's GraphCutSeamFinder."""
    from . import multiband_model as mb
    planes = graphcut_planes(layers, out_w, out_h, frames, maps, seam_frames, find_graphcut_cv2)
    C = mb._as3(frames[layers[0].cam]).shape[2]
    return _as_out(mb.blend_planes_cv2(planes, out_w, out_h, bands, C), frames, layers)
