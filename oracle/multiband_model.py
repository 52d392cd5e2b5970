"""ORACLE (test infrastructure, never imported by the product package).

Multi-band blend of the camera-weighted panorama (include/mcs.h mcs_plan_set_multiband): OpenCV's
``cv::detail::MultiBandBlender`` with ``CV_16S`` weights, fed with the per-camera planes of
``camera_weight_model.layer_planes`` on the layers of ``plan.flatten_chain``.  For each layer k with
a non-empty visible rectangle ``(x0, y0, x1, y1)`` (clipped to the panorama), ``v_k`` is the overwrite
sample there and ``w_k`` the same sample of the camera's weight map (no map = 255).  The panorama
with ``n`` bands is

    b = cv2.detail_MultiBandBlender(0, n, cv2.CV_16S); b.prepare((0, 0, out_w, out_h))
    for every such layer k, innermost first:  b.feed(v_k.astype(int16), w_k.astype(uint8), (x0, y0))
    dst, dst_mask = b.blend(None, None)
    out = saturate_u8(dst), 0 where dst_mask == 0

``feed`` takes 3-channel images only; the blend treats channels independently and shares the
weights, so a 1-channel panorama is channel 0 of the blend of the plane repeated three times, and a
4-channel one is channels 0-2 of one blend plus channel 2 of the blend of channels 1-3.

Two restatements, which the CPU tests hold equal:

``blend_cv2`` - the definition above, calling the cv2 class (the pin).

``blend`` - the same in numpy integers, step by step as OpenCV's CPU code runs it and as the kernels
of csrc/mcs_stitch_multiband.cu follow it: the band clamp and ROI padding of ``prepare``, the region
``feed`` keeps per camera, the ``CV_16S`` weight ``mask + (mask != 0)``, ``createLaplacePyr`` on int16,
the accumulation ``dst += (L * W) >> 8`` and ``W_sum += W`` with int16 wrap, the normalisation
``(L << 8) / (W_sum + 1)`` (division truncating toward zero), the collapse with saturating adds and
the crop with the zero mask.  ``pyr_down`` and ``pyr_up`` restate ``cv2.pyrDown`` / ``cv2.pyrUp`` on
int16: the 5-tap kernel [1 4 6 4 1], BORDER_REFLECT_101, ``(s + 128) >> 8`` and ``(s + 32) >> 6``.
"""
import math

import cv2
import numpy as np

from . import camera_weight_model

KERNEL = np.array([1, 4, 6, 4, 1], np.int64)


# ---- integer helpers ----------------------------------------------------------------------------
def sat16(a):
    return np.clip(a, -32768, 32767).astype(np.int64)


def wrap16(a):
    """Store to int16: the value modulo 2^16 (what the C cast to short does)."""
    return ((np.asarray(a, np.int64) + 32768) & 0xFFFF) - 32768


def trunc_div(a, b):
    """C integer division (toward zero) of int64 arrays."""
    a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
    q = np.abs(a) // np.abs(b)
    return np.where((a < 0) != (b < 0), -q, q)


def reflect(p, n, delta):
    """cv::borderInterpolate: BORDER_REFLECT (delta 0, ``fedcba|abcdef|fedcba``) or BORDER_REFLECT_101
    (delta 1, ``gfedcb|abcdefgh|gfedcba``) of the indices ``p`` into ``[0, n)``, repeated until inside."""
    p = np.array(p, np.int64, copy=True)
    if n == 1:
        return np.zeros_like(p)
    while True:
        lo, hi = p < 0, p >= n
        if not (lo.any() or hi.any()):
            return p
        p = np.where(lo, -p - 1 + delta, np.where(hi, n - 1 - (p - n) - delta, p))


def _as3(a):
    a = np.asarray(a)
    return a[:, :, None] if a.ndim == 2 else a


# ---- pyramids -----------------------------------------------------------------------------------
def pyr_down(a):
    """``cv2.pyrDown`` of an int16 image (H x W or H x W x C) to ((H + 1) // 2, (W + 1) // 2): the
    separable 5-tap sum over BORDER_REFLECT_101, one rounding ``(s + 128) >> 8``, saturation."""
    a3 = _as3(a).astype(np.int64)
    H, W = a3.shape[:2]
    dh, dw = (H + 1) // 2, (W + 1) // 2
    rows = np.zeros((dh, W, a3.shape[2]), np.int64)
    for j, k in enumerate(KERNEL):
        rows += k * a3[reflect(2 * np.arange(dh) + j - 2, H, 1)]
    s = np.zeros((dh, dw, a3.shape[2]), np.int64)
    for j, k in enumerate(KERNEL):
        s += k * rows[:, reflect(2 * np.arange(dw) + j - 2, W, 1)]
    out = sat16((s + 128) >> 8)
    return out[:, :, 0] if np.asarray(a).ndim == 2 else out


def _up_taps(n_dst, n_src):
    """Per destination index of ``pyr_up`` along one axis: three (source index, weight) pairs.  The
    source is zero-inserted to length 2 * n_src and convolved with the 5-tap kernel under
    BORDER_REFLECT_101 (which keeps the parity), so an even index takes 1 6 1 and an odd one 4 4."""
    idx, wt = [], []
    d = np.arange(n_dst)
    for m in (-2, -1, 0, 1, 2):
        j = reflect(d + m, 2 * n_src, 1)
        idx.append(j // 2)
        wt.append(np.where(j % 2 == 0, KERNEL[m + 2], 0))
    return idx, wt


def pyr_up(a, dsize=None):
    """``cv2.pyrUp`` of an int16 image to ``dsize = (w, h)`` (default twice the size; 2w - 1 is the
    same with the last column cut): ``(s + 32) >> 6``, saturation."""
    a3 = _as3(a).astype(np.int64)
    H, W = a3.shape[:2]
    dw, dh = (2 * W, 2 * H) if dsize is None else (int(dsize[0]), int(dsize[1]))
    ri, rw = _up_taps(dh, H)
    ci, cw = _up_taps(dw, W)
    rows = sum(w[:, None, None] * a3[i] for i, w in zip(ri, rw))
    s = sum(w[None, :, None] * rows[:, i] for i, w in zip(ci, cw))
    out = sat16((s + 32) >> 6)
    return out[:, :, 0] if np.asarray(a).ndim == 2 else out


def laplace_pyr(img, n):
    """``createLaplacePyr`` of an int16 image (the int16 branch): the pyrDown chain G_0..G_n, then
    L_i = G_i - pyrUp(G_{i+1}) saturated, L_n = G_n.  Returns ``(L, G)``."""
    G = [np.asarray(img, np.int64)]
    for _ in range(n):
        G.append(pyr_down(G[-1]))
    L = [sat16(G[i] - pyr_up(G[i + 1], (G[i].shape[1], G[i].shape[0]))) for i in range(n)] + [G[n]]
    return L, G


# ---- geometry of prepare / feed -----------------------------------------------------------------
def num_bands(requested, out_w, out_h):
    """``prepare``'s clamp: min(requested, ceil(log(max(w, h)) / log(2)))."""
    max_len = max(int(out_w), int(out_h))
    if max_len < 1:
        return 0
    return min(int(requested), int(math.ceil(math.log(max_len) / math.log(2.0))))


def roi_size(n, out_w, out_h):
    """``prepare``'s ROI, padded to multiples of 2^n."""
    s = 1 << n
    return out_w + (s - out_w % s) % s, out_h + (s - out_h % s) % s


def feed_region(rect, n, roi_w, roi_h):
    """``feed``'s region of an image at ``rect = (x0, y0, x1, y1)``: ``(tlx, tly, brx, bry)``.  The rectangle
    grows by ``3 * 2^n``, is clipped to the ROI, its corner aligned down and its size up to 2^n, and the
    region is shifted back inside at the right and bottom edges."""
    x0, y0, x1, y1 = rect
    s = 1 << n
    gap = 3 * s
    tlx, tly = max(0, x0 - gap), max(0, y0 - gap)
    brx, bry = min(roi_w, x1 + gap), min(roi_h, y1 + gap)
    tlx, tly = (tlx >> n) << n, (tly >> n) << n
    wd, ht = brx - tlx, bry - tly
    wd += (s - wd % s) % s
    ht += (s - ht % s) % s
    brx, bry = tlx + wd, tly + ht
    dx, dy = max(brx - roi_w, 0), max(bry - roi_h, 0)
    return tlx - dx, tly - dy, brx - dx, bry - dy


def bordered(v, w, rect, region):
    """Level 0 of one camera over its region: the image with a BORDER_REFLECT border (int16) and the
    ``CV_16S`` weight ``w + (w != 0)`` with a BORDER_CONSTANT 0 border."""
    x0, y0, x1, y1 = rect
    tlx, tly, brx, bry = region
    ry = reflect(np.arange(tly, bry) - y0, y1 - y0, 0)
    rx = reflect(np.arange(tlx, brx) - x0, x1 - x0, 0)
    img = _as3(v).astype(np.int64)[ry][:, rx]
    w16 = np.asarray(w, np.int64)
    w16 = w16 + (w16 != 0)
    wt = np.zeros((bry - tly, brx - tlx), np.int64)
    wt[y0 - tly:y1 - tly, x0 - tlx:x1 - tlx] = w16
    return img, wt


# ---- the blend ----------------------------------------------------------------------------------
def camera_planes(layers, out_w, out_h, frames, maps):
    """``[(rect, v, w)]`` of the layers with a non-empty visible rectangle, innermost first."""
    out = []
    for l in layers:
        rect, v, w = camera_weight_model.layer_planes(l, frames[l.cam], maps[l.cam], out_w, out_h)
        if rect[2] > rect[0] and rect[3] > rect[1]:
            out.append((rect, _as3(v), w))
    return out


def blend_planes(planes, out_w, out_h, bands, C):
    """The numpy restatement on ``[(rect, v (h x w x C), w (h x w))]``.  Returns ``(panorama H x W x C
    uint8, details)``; ``details`` holds the effective band count, the ROI, every camera's region,
    Gaussian, Laplacian and weight pyramids, the accumulated and normalised panorama pyramids, the
    summed weights and the collapsed levels, so that a kernel mismatch can be placed at a level."""
    n = num_bands(bands, out_w, out_h)
    RW, RH = roi_size(n, out_w, out_h)
    acc = [np.zeros((RH >> i, RW >> i, C), np.int64) for i in range(n + 1)]
    wsum = [np.zeros((RH >> i, RW >> i), np.int64) for i in range(n + 1)]
    cams = []
    for rect, v, w in planes:
        region = feed_region(rect, n, RW, RH)
        img, wt = bordered(v, w, rect, region)
        L, G = laplace_pyr(img, n)
        WG = [wt]
        for _ in range(n):
            WG.append(pyr_down(WG[-1]))
        tlx, tly, brx, bry = region
        for i in range(n + 1):
            ys, xs = slice(tly >> i, bry >> i), slice(tlx >> i, brx >> i)
            acc[i][ys, xs] = wrap16(acc[i][ys, xs] + ((L[i] * WG[i][..., None]) >> 8))
            wsum[i][ys, xs] = wrap16(wsum[i][ys, xs] + WG[i])
        cams.append(dict(rect=rect, region=region, G=G, L=L, W=WG))
    norm = [wrap16(trunc_div(acc[i] * 256, wsum[i][..., None] + 1)) for i in range(n + 1)]
    P = list(norm)
    for i in range(n, 0, -1):
        P[i - 1] = sat16(P[i - 1] + pyr_up(P[i], (RW >> (i - 1), RH >> (i - 1))))
    dst = P[0][:out_h, :out_w]
    mask = wsum[0][:out_h, :out_w] > 0
    out = np.where(mask[..., None], np.clip(dst, 0, 255), 0).astype(np.uint8)
    return out, dict(bands=n, roi=(RW, RH), cams=cams, acc=acc, wsum=wsum, norm=norm, restored=P)


def blend(layers, out_w, out_h, frames, maps, bands, details=False):
    """The numpy restatement on a plan's layers.  ``frames`` and ``maps`` are indexed by ``layer.cam``
    (``maps[cam]`` None = 255 everywhere).  The panorama is 2-D for 2-D frames."""
    C = _as3(frames[layers[0].cam]).shape[2]
    out, det = blend_planes(camera_planes(layers, out_w, out_h, frames, maps), out_w, out_h, bands, C)
    if np.asarray(frames[layers[0].cam]).ndim == 2:
        out = out[:, :, 0]
    return (out, det) if details else out


def cv2_blend3(planes, out_w, out_h, bands):
    """The cv2 class on 3-channel planes ``[(rect, v, w)]``: ``(int16 dst, u8 mask)``."""
    cv2.ocl.setUseOpenCL(False)
    b = cv2.detail_MultiBandBlender(0, int(bands), cv2.CV_16S)
    b.prepare((0, 0, int(out_w), int(out_h)))
    for (x0, y0, _, _), v, w in planes:
        b.feed(np.ascontiguousarray(v, np.int16), np.ascontiguousarray(w, np.uint8), (int(x0), int(y0)))
    return b.blend(None, None)


def blend_planes_cv2(planes, out_w, out_h, bands, C):
    """The definition on ``[(rect, v (h x w x C), w)]`` through the channel rule."""
    def run(sel):
        dst, mask = cv2_blend3([(r, v[:, :, sel], w) for r, v, w in planes], out_w, out_h, bands)
        dst = _as3(dst).astype(np.int64)
        return np.where((np.asarray(mask) > 0)[..., None], np.clip(dst, 0, 255), 0).astype(np.uint8)

    if not planes:
        return np.zeros((out_h, out_w, C), np.uint8)
    if C == 3:
        return run([0, 1, 2])
    if C == 1:
        return run([0, 0, 0])[:, :, :1]
    lo, hi = run([0, 1, 2]), run([1, 2, 3])
    return np.concatenate([lo, hi[:, :, 2:3]], axis=2)


def blend_cv2(layers, out_w, out_h, frames, maps, bands):
    """The definition, calling ``cv2.detail_MultiBandBlender``, on a plan's layers."""
    C = _as3(frames[layers[0].cam]).shape[2]
    out = blend_planes_cv2(camera_planes(layers, out_w, out_h, frames, maps), out_w, out_h, bands, C)
    return out[:, :, 0] if np.asarray(frames[layers[0].cam]).ndim == 2 else out
