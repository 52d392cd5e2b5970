"""ORACLE (test infrastructure, never imported by the product package).

Camera-weighted blend of the compositing chain (include/mcs.h mcs_plan_set_camera_weights).  The
reference has no such blend: it pastes each running canvas over the next camera
(PostScripts/Stitcher/StitcherClass.py:240-241), black wedges of the inner canvas included.  Here
every camera that sees an output pixel contributes, weighted by its own uint8 weight map ``W_k``
(one value per pixel of the camera's calibrated frame; no map = 255 everywhere), and the sum is
normalised per pixel.  Two restatements, which the CPU tests hold equal:

``blend`` - the layer-table model the kernel follows, on the layers of ``plan.flatten_chain``
(innermost first).  For output pixel p and layer k:

  reach_k(p)  p lies in the layer's visible rectangle (where canvas k, super-mode crops applied,
              appears in the panorama)
  v_k(p)      what the layer gives p in overwrite mode: the source pixel (COPY) or the fixed-point
              bilinear sample with BORDER_CONSTANT 0 (WARP, REMAP) of ``oracle/warp_model.py``
  w_k(p)      the same sample - coordinates, taps, rounding - of ``W_k``: exactly
              ``cv2.warpPerspective(W_k, cachedAH, ABSize)`` placed like the camera's image, so the
              weight fades over the camera's one-pixel border where taps fall outside the source
  contributors {k : reach_k(p) and w_k(p) > 0},  S = sum of their w_k
  out = (sum w_k * v_k + S // 2) // S per channel, 0 where S == 0

One contributor gives v_k whatever its weight; two equal weights give (v_0 + v_1 + 1) // 2.  Every
camera's sample is rounded to uint8 first, and the blend rounds once.

``chain`` - the same mode with plain cv2 calls, stage by stage as ``stitcher_ref.stitch_chain``
walks the reference: one (value, weight, reach) plane per camera, pasted at ``Bpts`` and cropped in
super mode with the canvas, the new camera and its map warped with ``cv2.warpPerspective``, the
planes combined at the end.
"""
import cv2
import numpy as np

from . import warp_model

LAYER_COPY = 0
LAYER_REMAP = 2
MAX_CONTRIBUTORS = 4


def _as3(a):
    a = np.asarray(a)
    return a[:, :, None] if a.ndim == 2 else a


def _coords(l, x0, y0, x1, y1):
    """1/32-px source coordinates of the layer over the output window [x0, x1) x [y0, y1)."""
    xs, ys = np.arange(x0 - l.ox, x1 - l.ox), np.arange(y0 - l.oy, y1 - l.oy)
    if l.kind == LAYER_COPY:
        return np.broadcast_to(xs[None, :] * 32, (len(ys), len(xs))), np.broadcast_to(ys[:, None] * 32, (len(ys), len(xs)))
    if l.kind == LAYER_REMAP:
        xy, frac = l.map
        f = np.zeros(xy.shape[:2], np.int64) if frac is None else np.asarray(frac).astype(np.int64)
        X = xy[..., 0].astype(np.int64) * 32 + (f & 31)
        Y = xy[..., 1].astype(np.int64) * 32 + ((f >> 5) & 31)
        return X[ys[:, None], xs[None, :]], Y[ys[:, None], xs[None, :]]
    Mi = warp_model.invert3x3(l.H)
    return warp_model.fixed_point_coords(np.zeros((3, 3)) if Mi is None else Mi, xs, ys)


def layer_planes(l, frame, wmap, out_w, out_h):
    """``((x0, y0, x1, y1), v, w)`` of one layer: its visible rectangle clipped to the panorama, the
    overwrite value there (uint8 h x w x C) and the sampled weight (int64 h x w)."""
    x0, y0, x1, y1 = [int(v) for v in l.rect]
    x0, y0, x1, y1 = max(0, x0), max(0, y0), min(out_w, x1), min(out_h, y1)
    x1, y1 = max(x0, x1), max(y0, y1)
    X, Y = _coords(l, x0, y0, x1, y1)
    src = _as3(frame)
    m = np.full(src.shape[:2], 255, np.uint8) if wmap is None else np.asarray(wmap, dtype=np.uint8)
    v, _ = warp_model.sample_fixed_point(src, np.asarray(X), np.asarray(Y))
    w, _ = warp_model.sample_fixed_point(m, np.asarray(X), np.asarray(Y))
    return (x0, y0, x1, y1), v, w[..., 0].astype(np.int64)


def combine(values, weights, reaches):
    """Normalised blend of full-panorama planes: ``values`` [K][H, W, C] uint8, ``weights`` [K][H, W],
    ``reaches`` [K][H, W] bool.  Returns ``(panorama, contributions per plane, most contributors)``."""
    H, W, C = values[0].shape
    num = np.zeros((H, W, C), np.int64)
    S = np.zeros((H, W), np.int64)
    count = np.zeros((H, W), np.int64)
    contrib = []
    for v, w, r in zip(values, weights, reaches):
        c = r & (np.asarray(w) > 0)
        wc = np.where(c, w, 0).astype(np.int64)
        num += wc[..., None] * v.astype(np.int64)
        S += wc
        count += c
        contrib.append(int(c.sum()))
    with np.errstate(divide="ignore", invalid="ignore"):
        out = np.where(S[..., None] > 0, (num + (S // 2)[..., None]) // np.maximum(S, 1)[..., None], 0)
    return out.astype(np.uint8), contrib, int(count.max()) if count.size else 0


def blend(layers, out_w, out_h, frames, maps):
    """The layer-table model.  ``frames`` and ``maps`` are indexed by ``layer.cam`` (``maps[cam]`` None =
    255 everywhere).  Returns ``(panorama, contributions per layer, most contributors of a pixel)``;
    the panorama is 2-D for 2-D frames."""
    C = _as3(frames[layers[0].cam]).shape[2]
    values, weights, reaches = [], [], []
    for l in layers:
        (x0, y0, x1, y1), v, w = layer_planes(l, frames[l.cam], maps[l.cam], out_w, out_h)
        V = np.zeros((out_h, out_w, C), np.uint8)
        Wt = np.zeros((out_h, out_w), np.int64)
        R = np.zeros((out_h, out_w), bool)
        V[y0:y1, x0:x1], Wt[y0:y1, x0:x1], R[y0:y1, x0:x1] = v, w, True
        values.append(V)
        weights.append(Wt)
        reaches.append(R)
    out, contrib, most = combine(values, weights, reaches)
    return (out[:, :, 0] if np.asarray(frames[layers[0].cam]).ndim == 2 else out), contrib, most


def chain(states, img_labels, images_dic, maps_by_label):
    """The chain restatement with cv2, stage by stage (oracle dict states, ``stitcher_ref``'s field
    names).  ``maps_by_label[label]``: uint8 map of the camera's frame or None.  Returns the panorama."""
    planes = chain_planes(states, img_labels, images_dic, maps_by_label)
    out, _, _ = combine(*zip(*planes))
    return out[:, :, 0] if np.asarray(images_dic[img_labels[0]]).ndim == 2 else out


def chain_planes(states, img_labels, images_dic, maps_by_label):
    """The per-camera ``(value, weight, reach)`` planes of ``chain``, each the size of the panorama."""
    def wmap(label):
        m = maps_by_label.get(label)
        return np.full(np.asarray(images_dic[label]).shape[:2], 255, np.uint8) if m is None else np.asarray(m, np.uint8)

    f0 = np.asarray(images_dic[img_labels[0]])
    planes = [(_as3(f0), wmap(img_labels[0]).astype(np.int64), np.ones(f0.shape[:2], bool))]
    for i, st in enumerate(states):
        if st["cachedAH"] is None:
            continue
        W, H = int(st["ABSize"][0]), int(st["ABSize"][1])
        bx, by = int(st["Bpts"][0][0]), int(st["Bpts"][0][1])
        moved = []
        for v, w, r in planes:   # StitcherClass.py:240-241: the running canvas is pasted at Bpts
            h, wd = r.shape
            V = np.zeros((H, W, v.shape[2]), np.uint8)
            Wt = np.zeros((H, W), np.int64)
            R = np.zeros((H, W), bool)
            V[by:by + h, bx:bx + wd], Wt[by:by + h, bx:bx + wd], R[by:by + h, bx:bx + wd] = v, w, r
            moved.append((V, Wt, R))
        label = img_labels[i + 1]
        warped = _as3(cv2.warpPerspective(np.asarray(images_dic[label]), st["cachedAH"], (W, H)))   # :239
        ww = cv2.warpPerspective(wmap(label), st["cachedAH"], (W, H)).astype(np.int64)
        moved.append((warped, ww, np.ones((H, W), bool)))
        if st["super_mode"]:   # :248-251
            ys, xs = slice(st["y_limits"][0], st["y_limits"][1]), slice(st["x_limits"][0], st["x_limits"][1])
            moved = [(v[ys, xs], w[ys, xs], r[ys, xs]) for v, w, r in moved]
        planes = moved
    return planes


def mulhi_div(n, S):
    """The kernel's division of ``n`` by ``S`` (2 <= S <= 4 * 255): ``__umulhi(n, ceil(2^32 / S))``."""
    m = (np.uint64(0xFFFFFFFF) // np.asarray(S, np.uint64)) + np.uint64(1)
    return (np.asarray(n, np.uint64) * m) >> np.uint64(32)
