"""Shared builders of the feather-blend tests: random rigs with trimmed super-mode crops, weight maps of every
kind, a cell-granularity model of the BAND tiles, and the tiled launcher's split rule restated."""
import os

import numpy as np

from multicamera_stitching_b200.plan import LAYER_COPY, flatten_chain, plan_paste
from oracle import feather_model, warp_model
from random_rigs import random_chain

SUPER_TRIM = (20, 12)   # super-mode crops this many pixels inside every stage canvas: they cut the pasted rectangles
CELL_W, CELL_H = 128, 16   # cell grid of the tiled kernel (MCS_CELL_W x MCS_CELL_H)
MAX_OVERLAYS = 2           # outer layers a BAND tile blends with (MCS_BAND_MAX_OVERLAYS)


def rig(seed):
    """``random_chain(seed)`` with trimmed super-mode crops, or None for a degenerate canvas."""
    return random_chain(seed, trim=SUPER_TRIM)


def stage_shapes(st, images, labels):
    """(height, width) of the canvas each stage pastes (its imageB): the shape of its weight map."""
    shapes = [tuple(images[labels[0]].shape[:2])]
    for sb in st.stitchers[:-1]:
        shapes.append(tuple(sb.result_shape()[:2]))
    return shapes


def make_maps(shapes, log2, kind, seed=0):
    """One uint8 weight map per stage of ``kind``: "random" 0..F with plateaus of F, "zero" / "one" / "fm1" /
    "full" constant 0 / 1 / F - 1 / F, "over" F + 1..255 where "random" has F, "checker" 0 / F, "mask" 0 / 1 (the
    weights of feather_log2 = 0)."""
    rng = np.random.default_rng(seed)
    F = 1 << log2
    maps = []
    for s in shapes:
        if kind in ("random", "over"):
            m = rng.integers(0, F + 1, size=s)
            plateau = rng.random(s) < 0.5
            m[plateau] = F if kind == "random" else rng.integers(F + 1, 256, size=int(plateau.sum()))
        elif kind == "checker":
            yy, xx = np.mgrid[0:s[0], 0:s[1]]
            m = np.where((xx + yy) % 2 == 0, 0, F)
        elif kind == "mask":
            m = (rng.random(s) < 0.7).astype(np.int64)
        else:
            m = np.full(s, {"zero": 0, "one": 1, "fm1": F - 1, "full": F}[kind])
        maps.append(np.ascontiguousarray(m, dtype=np.uint8))
    return maps


def layer_maps(flat, maps):
    """Weight maps in the plan's layer order (entry k = the paste of stage k - 1 over layer k's warp)."""
    out = [None] * len(flat.layers)
    if maps is not None:
        for k, l in enumerate(flat.layers):
            if l.cam >= 1:
                out[k] = maps[l.cam - 1]
    return out


def is_cut(flat):
    """A super-mode crop cut a pasted rectangle: distances run to the pasted edges (weight-map path only)."""
    paste = plan_paste(flat)
    return any(tuple(paste[k]) != tuple(l.rect) for k, l in enumerate(flat.layers[:-1])
               if l.rect[2] > l.rect[0] and l.rect[3] > l.rect[1])


def _tiles(flat):
    """(layer, cx0, y0, c0, c1, h) of every tile owned by a layer, on the 128 x 16 grid anchored at column 0,
    in the order mcs_tiles.cu cuts the rings."""
    out, inner = [], None
    for k, l in enumerate(flat.layers):
        r = tuple(int(v) for v in l.rect)
        if r[2] <= r[0] or r[3] <= r[1]:
            continue
        if inner is None:
            pieces = [r]
        else:
            pieces = [(r[0], r[1], r[2], inner[1]), (r[0], inner[3], r[2], r[3]),
                      (r[0], inner[1], inner[0], inner[3]), (inner[2], inner[1], r[2], inner[3])]
        for x0, y0, x1, y1 in pieces:
            if x1 <= x0 or y1 <= y0:
                continue
            for y in range(y0, y1, CELL_H):
                for i in range(x0 // CELL_W, (x1 - 1) // CELL_W + 1):
                    cx0 = i * CELL_W
                    out.append((k, cx0, y, max(x0, cx0) - cx0, min(x1, cx0 + CELL_W) - cx0, min(CELL_H, y1 - y)))
        inner = r
    return out


def _touched(l, W, H):
    """Where layer ``l``'s warp reads at least one tap inside its source, over the whole panorama."""
    if l.kind == LAYER_COPY:
        m = np.zeros((H, W), bool)
        x0, y0, x1, y1 = l.rect
        m[y0:y1, x0:x1] = True
        return m
    Mi = warp_model.invert3x3(np.asarray(l.H, dtype=np.float64))
    X, Y = warp_model.fixed_point_coords(Mi, np.arange(W) - l.ox, np.arange(H) - l.oy)
    sx, sy = np.clip(X >> 5, -32768, 32767), np.clip(Y >> 5, -32768, 32767)
    h, w = l.src_hw
    return ((((sx >= 0) & (sx < w)) | ((sx + 1 >= 0) & (sx + 1 < w))) &
            (((sy >= 0) & (sy < h)) | ((sy + 1 >= 0) & (sy + 1 < h))))


def band_tiles(flat, log2, maps=None):
    """The BAND tiles of the fused form, at cell granularity, from the specification: per tile of layer j, the
    outer layers k > j with a pixel of the tile where stage k blends (weight below F, layer k's warp touches its
    source).  Returns ``[(number of outer layers, zero base)]`` over the tiles with at least one; zero base = the
    owner's warp touches nothing in the tile (its value so far is 0).  The fused form exists when no tile has
    more than MAX_OVERLAYS."""
    F = 1 << log2
    W, H = flat.out_w, flat.out_h
    paste = plan_paste(flat)
    lmaps = layer_maps(flat, maps)
    touched = [_touched(l, W, H) for l in flat.layers]
    blends = [None]
    for k in range(1, len(flat.layers)):
        x0, y0, x1, y1 = (int(v) for v in paste[k - 1])
        a = np.full((H, W), F, np.int64)     # outside the pasted rectangle: nothing blends
        if x1 > x0 and y1 > y0:
            if lmaps[k] is not None:
                wmap = np.minimum(lmaps[k].astype(np.int64), F)
            else:
                wmap = feather_model.ramp_weights((y1 - y0, x1 - x0), log2).astype(np.int64)
            vx0, vy0, vx1, vy1 = max(0, x0), max(0, y0), min(W, x1), min(H, y1)
            if vx1 > vx0 and vy1 > vy0:
                a[vy0:vy1, vx0:vx1] = wmap[vy0 - y0:vy1 - y0, vx0 - x0:vx1 - x0]
        blends.append(touched[k] & (a < F))
    out = []
    for j, cx0, y, c0, c1, h in _tiles(flat):
        win = (slice(y, y + h), slice(cx0 + c0, cx0 + c1))
        n = sum(1 for k in range(j + 1, len(flat.layers)) if blends[k][win].any())
        if n:
            out.append((n, not touched[j][win].any()))
    return out


def plan_flat(st, images, labels):
    return flatten_chain(st.stitchers, [images[l].shape for l in labels])


def split_rule(stats, ctas_per_sm, n_sm, n_frames):
    """``(split, split_first, split_end)`` of mcs_launch_tiled: the resampled tiles [split_first, split_end) of the
    table (BAND, FAST, WARP, in that order) are cut into ``split`` chunks each.  ``stats`` = ``tiled_stats()`` (its
    frame block follows $MCS_TILED_FRAME_BLOCK), $MCS_TILED_SPLIT overrides the factor."""
    fb = min(stats["frame_block"], n_frames)
    nf_last = n_frames - (-(-n_frames // fb) - 1) * fb
    grid = min(n_sm * ctas_per_sm, stats["tiles"] * fb)
    split_end = stats["band"] + stats["fast"] + stats["warp"]
    split = 4 if fb >= 16 else 1
    env = os.environ.get("MCS_TILED_SPLIT")
    if env is not None:
        split = int(env) if int(env) > 1 and fb >= int(env) else 1
    if split > 1 and nf_last < split:
        split = 1          # a last block shorter than the split factor: chunks without frames, no split
    split_first = max(0, split_end - 2 * grid) if split > 1 else split_end
    return split, split_first, split_end
