"""The tiled kernel's four-pixel group path (FAST tiles, ``mcs_tile_fast_kernel`` in csrc/mcs_tiles.cu and
``sample_group`` / ``fast_frames`` in csrc/mcs_stitch_tiled.cu) against cv2, on the geometries that select it.

A 3-channel WARP tile becomes a FAST tile when, in each of its eight warps, at most 12 owned pixels fall off the
group template (four adjacent output pixels whose taps lie 3 bytes apart in one source row pair).  That happens
at near-unit scale only: sub-pixel translations, scales of 0.98-1.04, rotations under a degree - cameras side by
side, a pre-warped bird's-eye view, a mild undistortion.  The synthetic rigs step 1.01-1.13 source pixels per
output pixel and hardly reach it, so these tests build such geometries on purpose and check, besides bit-exact
output, that the path they target really ran: the tile counts of ``tiled_stats()`` against ``classify``, a numpy
restatement of the plan-time classification rule (the CPU test at the end keeps the chosen geometries on the
path).
"""
import math

import numpy as np
import pytest

from helpers import compare_u8
from multicamera_stitching_b200.plan import LAYER_COPY, LAYER_WARP, FlatPlan, Layer, flatten_chain
from oracle import stitcher_ref, warp_model

CELL_W, CELL_H = 128, 16    # cell grid of the tiled kernel (MCS_CELL_W x MCS_CELL_H)
FAST_LIMIT = 12             # default of $MCS_TILED_FAST_MAX: off-template pixels a warp may have


# ---- CPU model of the classification ---------------------------------------------------------------------------
def _ring(outer, inner):
    """outer minus inner (inner inside outer) as up to four rectangles, the way mcs_tiles.cu cuts them."""
    if outer[2] <= outer[0] or outer[3] <= outer[1]:
        return []
    if inner is None:
        return [outer]
    ox0, oy0, ox1, oy1 = outer
    ix0, iy0, ix1, iy1 = inner
    return [(ox0, oy0, ox1, iy0), (ox0, iy1, ox1, oy1), (ox0, iy0, ix0, iy1), (ix1, iy0, ox1, iy1)]


def _tiles(flat):
    """(layer, cx0, y0, c0, c1, h) of every tile owned by a layer, on the 128 x 16 grid anchored at column 0."""
    out, inner = [], None
    for k, l in enumerate(flat.layers):
        r = tuple(int(v) for v in l.rect)
        if r[2] <= r[0] or r[3] <= r[1]:
            continue
        for x0, y0, x1, y1 in _ring(r, inner):
            if x1 <= x0 or y1 <= y0:
                continue
            for y in range(y0, y1, CELL_H):
                for i in range(x0 // CELL_W, (x1 - 1) // CELL_W + 1):
                    cx0 = i * CELL_W
                    out.append((k, cx0, y, max(x0, cx0) - cx0, min(x1, cx0 + CELL_W) - cx0, min(CELL_H, y1 - y)))
        inner = r
    return out


def classify(flat, limit=FAST_LIMIT, pitch_words=32):
    """Tile counts of a 3-channel plan without blending, as ``mcs_plan_build_tiles`` classifies its WARP tiles.

    Per cell (every owned pixel, taps clamped to [-2, src]): the box origin (16-byte aligned byte column of the
    smallest tap column, smallest tap row) and the layer's box pitch.  Per group of four cell columns: the
    anchor bA = box byte offset of the first owned pixel's tap minus 3 bytes per column before it; a pixel fits
    when the anchor is addressable (bA >= 0) and its tap sits at bA + 3 j.  Per warp (cell rows w and w + 8):
    the pixels that do not fit.  A cell is FAST when no warp has more than ``limit``, with one general pass per
    32 of the busiest warp's."""
    C = flat.channels
    assert C == 3
    cells = []
    for k, cx0, y0, c0, c1, h in _tiles(flat):
        l = flat.layers[k]
        if l.kind == LAYER_COPY:
            cells.append(("copy", k, None))
            continue
        assert l.kind == LAYER_WARP
        src_h, src_w = (int(v) for v in l.src_hw)
        Mi = warp_model.invert3x3(l.H)
        Mi = np.zeros((3, 3)) if Mi is None else Mi
        X, Y = warp_model.fixed_point_coords(Mi, np.arange(cx0, cx0 + CELL_W) - l.ox, np.arange(y0, y0 + CELL_H) - l.oy)
        rsx, rsy = np.clip(X >> 5, -32768, 32767), np.clip(Y >> 5, -32768, 32767)
        cols, rows = np.arange(CELL_W)[None, :], np.arange(CELL_H)[:, None]
        own = (cols >= c0) & (cols < c1) & (rows < h)
        inside = (((rsx >= 0) & (rsx < src_w)) | ((rsx + 1 >= 0) & (rsx + 1 < src_w))) & \
                 (((rsy >= 0) & (rsy < src_h)) | ((rsy + 1 >= 0) & (rsy + 1 < src_h)))
        if not (inside & own).any():
            cells.append(("zero", k, None))
            continue
        sx, sy = np.clip(rsx, -2, src_w), np.clip(rsy, -2, src_h)
        bx = 4 * ((int(sx[own].min()) * C) // 16)            # box origin in words, 16-byte aligned
        by = int(sy[own].min())
        need_w = ((int(sx[own].max()) + 2) * C + 3) // 4 - bx + 1
        cells.append(("warp", k, dict(sx=sx, sy=sy, own=own, bx=bx, by=by, need_w=need_w)))
    bw4 = {}
    for cls, k, d in cells:
        if cls == "warp":
            bw4[k] = max(bw4.get(k, 0), d["need_w"])
    out = dict(fast=0, warp=0, copy=0, zero=0, fast_passes=0, max_off=[])
    for cls, k, d in cells:
        if cls != "warp":
            out[cls] += 1
            continue
        sp = -(-bw4[k] // pitch_words) * pitch_words * 4
        b = (d["sy"] - d["by"]) * sp + d["sx"] * C - 4 * d["bx"]
        own = d["own"].reshape(CELL_H, 32, 4)
        b = b.reshape(CELL_H, 32, 4)
        j0 = np.argmax(own, axis=2)                           # first owned pixel of each group
        bA = np.take_along_axis(b, j0[..., None], axis=2)[..., 0] - 3 * j0
        fit = own & (bA >= 0)[..., None] & (b == bA[..., None] + 3 * np.arange(4))
        off = (own & ~fit).sum(axis=(1, 2))                  # per cell row
        per_warp = np.minimum(off[:8] + off[8:], 255)
        mx = int(per_warp.max())
        out["max_off"].append(mx)
        if mx <= limit:
            out["fast"] += 1
            out["fast_passes"] = max(out["fast_passes"], -(-mx // 32))
        else:
            out["warp"] += 1
    return out


# ---- geometries -------------------------------------------------------------------------------------------------
# A = panorama -> camera (what the kernel evaluates); the layer stores the forward camera -> panorama map.
def A_translate(tx, ty):
    return np.array([[1.0, 0.0, tx], [0.0, 1.0, ty], [0.0, 0.0, 1.0]])


def A_scale(s, cx=0.0, cy=0.0):
    return np.array([[s, 0.0, cx * (1 - s)], [0.0, s, cy * (1 - s)], [0.0, 0.0, 1.0]])


def A_rot(deg, cx=320.0, cy=180.0):
    c, s = math.cos(math.radians(deg)), math.sin(math.radians(deg))
    return np.array([[c, -s, cx - c * cx + s * cy], [s, c, cy - s * cx - c * cy], [0.0, 0.0, 1.0]])


def single_layer(A, src_hw, out_w, out_h, channels=3):
    """One WARP layer covering the whole panorama: ``cv2.warpPerspective(src, inv(A), (out_w, out_h))``."""
    M = np.linalg.inv(A)
    return FlatPlan([Layer(0, LAYER_WARP, M, 0, 0, (0, 0, out_w, out_h), tuple(src_hw))], out_w, out_h, channels,
                    3 if channels > 1 else 2)


def translation_chain(n, h, w, steps, xoffset=0, yoffset=0):
    """Oracle states (dicts) of an n-camera chain in which camera k + 1 sits ``steps[k]`` = (tx, ty) pixels from
    the running canvas: pure translations, sub-pixel ones put every camera on the group path."""
    states, shapeB = [], (h, w, 3)
    for k in range(n - 1):
        st = stitcher_ref.new_state(sid=str(k))
        stitcher_ref.geometry_from_homography(st, A_translate(*steps[k]), (h, w, 3), shapeB, xoffset, yoffset)
        states.append(st)
        shapeB = (st["ABSize"][1], st["ABSize"][0], 3)
    return states


def chain_flat(states, h, w):
    return flatten_chain(states, [(h, w, 3)] * (len(states) + 1))


# Sub-pixel translations: the x phase runs through all 32 fractions, the y phase through (7 i) % 32.
PHASES = [(i, (7 * i) % 32) for i in range(32)]
PHASE_SRC = (80, 272)           # source of the 256 x 64 phase plans: covers every tap, no clamping


def phase_A(i, j):
    return A_translate(5 + i / 32.0, 3 + j / 32.0)


# 640 x 360 -> 640 x 360 geometries whose general lists are not empty (panorama -> camera)
GENERAL = {
    "scale1.005": A_scale(1.005),
    "scale0.98": A_scale(0.98),
    "scale1.02": A_scale(1.02),
    "scale1.04": A_scale(1.04),
    "rot0.3": A_rot(0.3),
    "rot1": A_rot(1.0),
}
# (source h x w, panorama w x h, tx, ty): translations that leave clamped taps (2+ pixels outside the source) on all
# four sides; a few clamped columns fit a FAST cell's general lists, twenty do not (the last one mixes the classes)
BORDERS = [((150, 250), (256, 160), -3.37, -2.71), ((150, 250), (256, 160), -2.84, -3.03),
           ((150, 250), (264, 168), -6.37, -5.71), ((200, 460), (512, 240), -20.37, -13.71)]


def _clamped_sides(flat):
    """Sides (left, right, top, bottom) of the source beyond which some pixel's taps are clamped."""
    l = flat.layers[0]
    X, Y = warp_model.fixed_point_coords(warp_model.invert3x3(l.H), np.arange(flat.out_w), np.arange(flat.out_h))
    src_h, src_w = l.src_hw
    return ((X >> 5) < -2).any(), ((X >> 5) > src_w).any(), ((Y >> 5) < -2).any(), ((Y >> 5) > src_h).any()
# two-camera chains whose inner rectangle ends at a column = xoffset (mod 4) and whose camera 1 samples source
# column 336 = 16 * 21 there: the group holding that column has its first owned tap at the 16-byte aligned box
# start, so its anchor (3 * j0 bytes further left) is not addressable
ANCHOR_STEP = (303.37, 5.71)


def _unanchored(flat):
    """Groups of FAST-eligible cells whose anchor lies left of the box start (model of ``anchored = bA >= 0``)."""
    n = 0
    for k, cx0, y0, c0, c1, h in _tiles(flat):
        l = flat.layers[k]
        if l.kind != LAYER_WARP:
            continue
        src_h, src_w = (int(v) for v in l.src_hw)
        X, Y = warp_model.fixed_point_coords(warp_model.invert3x3(l.H), np.arange(cx0, cx0 + CELL_W) - l.ox,
                                             np.arange(y0, y0 + CELL_H) - l.oy)
        sx, sy = np.clip(X >> 5, -2, src_w), np.clip(Y >> 5, -2, src_h)
        cols, rows = np.arange(CELL_W)[None, :], np.arange(CELL_H)[:, None]
        own = (cols >= c0) & (cols < c1) & (rows < h)
        if not own.any():
            continue
        bx3 = 16 * ((int(sx[own].min()) * 3) // 16)
        by = int(sy[own].min())
        # bA < 0 needs the first owned tap in the box's first row, less than 3 * j0 bytes after its start
        g_own = own.reshape(CELL_H, 32, 4)
        j0 = np.argmax(g_own, axis=2)
        first = np.take_along_axis((sx * 3 - bx3).reshape(CELL_H, 32, 4), j0[..., None], axis=2)[..., 0]
        top = np.take_along_axis((sy == by).reshape(CELL_H, 32, 4), j0[..., None], axis=2)[..., 0]
        n += int((g_own.any(axis=2) & top & (first < 3 * j0)).sum())
    return n


# ---- GPU helpers --------------------------------------------------------------------------------------------------
def _noise(shape, seed):
    return np.random.default_rng(seed).integers(0, 256, size=shape, dtype=np.uint8)


def _compiled(flat, device, monkeypatch=None, **env):
    """A fresh plan (the $MCS_TILED_* knobs are read when the plan is built)."""
    from multicamera_stitching_b200.engine import CompiledPlan
    if env:
        for k, v in env.items():
            monkeypatch.setenv(k, str(v))
    try:
        return CompiledPlan(flat, device)
    finally:
        for k in env:
            monkeypatch.delenv(k)


def _run(plan, src, device, variant=2, out=None, n_frames=None):
    import torch
    plan.handle.force_variant(variant)
    try:
        res = plan.run([torch.from_numpy(np.ascontiguousarray(src)).to(device)], out=out, n_frames=n_frames)
        assert plan.handle.last_variant() == variant
    finally:
        plan.handle.force_variant(0)
    return res


def _warp_ref(src, flat):
    import cv2
    l = flat.layers[0]
    return cv2.warpPerspective(src, l.H, (flat.out_w, flat.out_h))


def _assert_counts(plan, model):
    s = plan.handle.tiled_stats()
    got = {k: s[k] for k in ("fast", "warp", "zero", "fast_passes")}
    want = {k: model[k] for k in ("fast", "warp", "zero", "fast_passes")}
    assert got == want, (got, want)
    return s


# ---- 1. every sub-pixel phase ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_every_subpixel_phase_of_a_translation(cuda_device):
    src = _noise(PHASE_SRC + (3,), 1)
    for i, j in PHASES:
        flat = single_layer(phase_A(i, j), PHASE_SRC, 256, 64)
        plan = _compiled(flat, cuda_device)
        s = _assert_counts(plan, classify(flat))
        assert s["fast"] == 8 and s["warp"] == 0 and s["fast_passes"] == 0, (i, j, s)
        ref = _warp_ref(src, flat)
        assert compare_u8(_run(plan, src, cuda_device).cpu().numpy(), ref) == (0, 1.0), (i, j)
        assert compare_u8(_run(plan, src, cuda_device, variant=1).cpu().numpy(), ref) == (0, 1.0), (i, j)


@pytest.mark.gpu
def test_all_phases_inside_one_near_unit_scale_plan(cuda_device):
    flat = single_layer(GENERAL["scale1.005"], (360, 640), 640, 360)
    X, Y = warp_model.fixed_point_coords(warp_model.invert3x3(flat.layers[0].H), np.arange(640), np.arange(360))
    assert len(np.unique(X & 31)) == 32 and len(np.unique(Y & 31)) == 32
    src = _noise((360, 640, 3), 2)
    plan = _compiled(flat, cuda_device)
    s = _assert_counts(plan, classify(flat))
    assert s["warp"] == 0 and s["fast_passes"] == 1
    assert compare_u8(_run(plan, src, cuda_device).cpu().numpy(), _warp_ref(src, flat)) == (0, 1.0)


# ---- 2. general lists -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GENERAL))
def test_general_lists(cuda_device, monkeypatch, name):
    flat = single_layer(GENERAL[name], (360, 640), 640, 360)
    src = _noise((360, 640, 3), 3)
    ref = _warp_ref(src, flat)
    plan = _compiled(flat, cuda_device)
    s = _assert_counts(plan, classify(flat))
    assert s["fast"] > 0 and s["fast_passes"] == 1
    if name in ("scale1.02", "scale1.04"):
        assert s["warp"] > 0
    got = _run(plan, src, cuda_device).cpu().numpy()
    assert compare_u8(got, ref) == (0, 1.0)
    # only template-perfect tiles
    plan0 = _compiled(flat, cuda_device, monkeypatch, MCS_TILED_FAST_MAX=0)
    _assert_counts(plan0, classify(flat, limit=0))
    assert compare_u8(_run(plan0, src, cuda_device).cpu().numpy(), ref) == (0, 1.0)
    # per-pixel descriptors only, and the gather kernel: the same bytes
    plain = _compiled(flat, cuda_device, monkeypatch, MCS_TILED_FAST=0)
    assert plain.handle.tiled_stats()["fast"] == 0
    assert np.array_equal(_run(plain, src, cuda_device).cpu().numpy(), got)
    assert np.array_equal(_run(plain, src, cuda_device, variant=1).cpu().numpy(), got)


@pytest.mark.gpu
def test_two_general_passes(cuda_device, monkeypatch):
    flat = single_layer(GENERAL["scale1.04"], (360, 640), 640, 360)
    src = _noise((360, 640, 3), 4)
    plan = _compiled(flat, cuda_device, monkeypatch, MCS_TILED_FAST_MAX=64)
    s = _assert_counts(plan, classify(flat, limit=64))
    assert s["fast_passes"] == 2
    assert compare_u8(_run(plan, src, cuda_device).cpu().numpy(), _warp_ref(src, flat)) == (0, 1.0)


# ---- 3. source borders, unaddressable anchors ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("src_hw,out_wh,tx,ty", BORDERS)
def test_clamped_taps_on_all_four_sides(cuda_device, src_hw, out_wh, tx, ty):
    flat = single_layer(A_translate(tx, ty), src_hw, *out_wh)
    src = _noise(src_hw + (3,), 5)
    plan = _compiled(flat, cuda_device)
    s = _assert_counts(plan, classify(flat))
    assert s["fast"] > 0
    ref = _warp_ref(src, flat)
    assert compare_u8(_run(plan, src, cuda_device).cpu().numpy(), ref) == (0, 1.0)
    assert compare_u8(_run(plan, src, cuda_device, variant=1).cpu().numpy(), ref) == (0, 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("xoffset", [1, 2, 3])
def test_anchor_left_of_the_box_start(cuda_device, xoffset):
    from multicamera_stitching_b200 import Stitcher
    h, w = 120, 640
    states = translation_chain(2, h, w, [ANCHOR_STEP], xoffset, 4)
    images = {"CAM1": _noise((h, w, 3), 6), "CAM2": _noise((h, w, 3), 7)}
    st = Stitcher(images)
    st.stitchers[0].set_homography(A_translate(*ANCHOR_STEP), (h, w, 3), (h, w, 3), xoffset, 4)
    plan = st.plan([(h, w, 3)] * 2, cuda_device)
    flat = chain_flat(states, h, w)
    assert flat.layers[0].rect[2] % 4 == xoffset and _unanchored(flat) > 0
    s = _assert_counts(plan, classify(flat))
    assert s["fast"] > 0
    ref = stitcher_ref.stitch_chain(states, ["CAM1", "CAM2"], images)
    assert compare_u8(st.stitch(images), ref) == (0, 1.0)
    assert plan.handle.last_variant() == 2


# ---- 4. output layouts: use_fast and phase_moves ---------------------------------------------------------------------
def _layout_case(plan, srcs, device, pitch, offset, fstride):
    """Composite len(srcs) frames into a sentinel-filled buffer with this row pitch, base offset and frame stride;
    returns (frames, bytes outside the view that were written)."""
    import torch
    F = len(srcs)
    row = plan.out_w * 3
    total = offset + (F - 1) * fstride + plan.out_h * pitch + 64
    buf = torch.full((total,), 0xAB, dtype=torch.uint8, device=device)
    out = torch.as_strided(buf, (F, plan.out_h, plan.out_w, 3), (fstride, pitch, 3, 1), storage_offset=offset)
    batch = torch.from_numpy(np.stack(srcs)).to(device)
    plan.handle.force_variant(2)
    try:
        plan.run([batch], out=out, n_frames=F)
        assert plan.handle.last_variant() == 2
    finally:
        plan.handle.force_variant(0)
    flat = buf.cpu().numpy()
    mask = np.zeros(total, bool)
    for f in range(F):
        for y in range(plan.out_h):
            a = offset + f * fstride + y * pitch
            mask[a:a + row] = True
    return out.cpu().numpy(), int((flat[~mask] != 0xAB).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("out_w,pitch,offset,fstride_pad,F", [
    (253, 759, 0, 0, 1),    # dense 759-byte rows: the group path is off, per-pixel descriptors serve the FAST tiles
    (253, 760, 0, 0, 1),    # 4-byte multiple, 8 mod 16: group path on, the 16-byte phase moves from row to row
    (253, 764, 0, 0, 1),    # 12 mod 16
    (253, 768, 0, 0, 1),    # 16-byte multiple
    (253, 896, 0, 0, 1),    # 128-byte multiple
    (256, 768, 4, 0, 1),    # base +4: group path on
    (256, 768, 1, 0, 1),    # base +1 / +2 / +3: group path off
    (256, 768, 2, 0, 1),
    (256, 768, 3, 0, 1),
    (256, 768, 0, 4, 5),    # frame stride 4 / 8 / 12 mod 16: one fast_frames call per frame
    (256, 768, 0, 8, 5),
    (256, 768, 4, 12, 19),
    (256, 768, 0, 2, 5),    # frame stride 2 mod 4: group path off
    (253, 760, 0, 0, 3),    # a batch of pitch 8 mod 16 rows, frame stride 64 x 760 = 0 mod 16
])
def test_output_layouts(cuda_device, out_w, pitch, offset, fstride_pad, F):
    flat = single_layer(phase_A(13, 11), PHASE_SRC, out_w, 64)
    plan = _compiled(flat, cuda_device)
    s = _assert_counts(plan, classify(flat))
    assert s["fast"] > 0 and s["warp"] == 0
    srcs = [_noise(PHASE_SRC + (3,), 10 + f) for f in range(F)]
    got, stray = _layout_case(plan, srcs, cuda_device, pitch, offset, 64 * pitch + fstride_pad)
    assert stray == 0
    for f in range(F):
        assert compare_u8(got[f], _warp_ref(srcs[f], flat)) == (0, 1.0), f


# ---- 5. work split ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("frame_block", [None, 4])
def test_split_fast_tiles(cuda_device, monkeypatch, frame_block):
    """Eight FAST tiles: fewer than two per CTA, so with 16+ frames per block every one of them is cut into four
    chunks (split_first = 0); with $MCS_TILED_FRAME_BLOCK=4 and $MCS_TILED_SPLIT=4 into chunks of one frame."""
    import torch
    flat = single_layer(phase_A(21, 3), PHASE_SRC, 256, 64)
    env = {} if frame_block is None else dict(MCS_TILED_FRAME_BLOCK=frame_block)
    plan = _compiled(flat, cuda_device, monkeypatch, **env)
    s = _assert_counts(plan, classify(flat))
    assert s["fast"] == 8 and s["warp"] == 0
    if frame_block:
        monkeypatch.setenv("MCS_TILED_SPLIT", "4")
    srcs = [_noise(PHASE_SRC + (3,), 100 + f) for f in range(65)]
    refs = [_warp_ref(x, flat) for x in srcs]
    dev = torch.from_numpy(np.stack(srcs)).to(cuda_device)
    for F in (1, 3, 16, 17, 64, 65):
        plan.handle.force_variant(2)
        try:
            got = plan.run([dev[:F]], n_frames=F).cpu().numpy()
            assert plan.handle.last_variant() == 2
        finally:
            plan.handle.force_variant(0)
        for f in range(F):
            assert compare_u8(got[f], refs[f]) == (0, 1.0), (F, f)


# ---- 6. run-time box pitch ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_run_time_box_pitch(cuda_device, monkeypatch):
    flat = single_layer(phase_A(7, 17), PHASE_SRC, 256, 64)
    src = _noise(PHASE_SRC + (3,), 8)
    default = _compiled(flat, cuda_device)
    plan = _compiled(flat, cuda_device, monkeypatch, MCS_TILED_PITCH_WORDS=4)
    s = _assert_counts(plan, classify(flat, pitch_words=4))
    assert s["fast"] == 8
    assert s["box_bytes"] != default.handle.tiled_stats()["box_bytes"]
    assert compare_u8(_run(plan, src, cuda_device).cpu().numpy(), _warp_ref(src, flat)) == (0, 1.0)


# ---- 7. blend modes ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("log2", [2, 3, 4])
def test_band_and_fast_tiles_in_one_launch(cuda_device, log2):
    from multicamera_stitching_b200 import Stitcher
    from oracle import feather_model
    h, w = 96, 320
    steps = [(200.37, 3.71), (150.84, -4.29)]
    states = translation_chain(3, h, w, steps, 5, 6)
    labels = ["CAM1", "CAM2", "CAM3"]
    images = {l: _noise((h, w, 3), 20 + k) for k, l in enumerate(labels)}
    st = Stitcher(images)
    shapeB = (h, w, 3)
    for k, step in enumerate(steps):
        st.stitchers[k].set_homography(A_translate(*step), (h, w, 3), shapeB, 5, 6)
        shapeB = st.stitchers[k].result_shape()
    st.feather_log2 = log2
    got = st.stitch(images)
    assert compare_u8(got, feather_model.feather_chain(states, labels, images, log2)) == (0, 1.0)
    plan = st.plan([(h, w, 3)] * 3, cuda_device)
    s = plan.handle.tiled_stats()
    assert s["band"] > 0 and s["fast"] > 0 and s["band_fused"] == 1, s
    assert plan.handle.last_variant() == 4
    rng = np.random.default_rng(log2)
    F = 1 << log2
    maps, shapeB = [], (h, w)
    for sb in st.stitchers:
        m = rng.integers(0, F + 1, size=shapeB).astype(np.uint8)
        m[rng.random(shapeB) < 0.6] = F
        maps.append(m)
        shapeB = sb.result_shape()[:2]
    st.blend_weights = maps
    got = st.stitch(images)
    assert compare_u8(got, feather_model.feather_chain(states, labels, images, log2, maps)) == (0, 1.0)
    plan = st.plan([(h, w, 3)] * 3, cuda_device)
    s = plan.handle.tiled_stats()
    assert s["band"] > 0 and s["fast"] > 0 and s["band_fused"] == 1, s
    assert plan.handle.last_variant() == 4


# ---- 8. other inputs ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("strength", [0.05, 0.2])
def test_weak_undistortion(cuda_device, strength):
    import cv2
    from multicamera_stitching_b200 import prewarp
    from multicamera_stitching_b200.plan import LAYER_REMAP
    from test_oracle_prewarp import camera
    h, w = 360, 640
    mtx, dist = camera(h, w, strength)
    img = _noise((h, w, 3), 30)
    maps = prewarp.undistort_maps(mtx, dist, (w, h))
    flat = FlatPlan([Layer(0, LAYER_REMAP, None, 0, 0, (0, 0, w, h), (h, w), maps)], w, h, 3, 3)
    plan = _compiled(flat, cuda_device)
    s = plan.handle.tiled_stats()
    assert s["fast"] > 0, s
    assert compare_u8(_run(plan, img, cuda_device).cpu().numpy(), cv2.undistort(img, mtx, dist)) == (0, 1.0)
    assert compare_u8(prewarp.undistort(img, mtx, dist), cv2.undistort(img, mtx, dist)) == (0, 1.0)


@pytest.mark.gpu
def test_rows_that_need_padding(cuda_device):
    """131-pixel BGR rows (393 bytes) go through zero-padded scratch rows; the taps right of the last column read
    the pad bytes."""
    flat = single_layer(A_translate(3.37, 2.59), (80, 131), 128, 64)
    src = _noise((80, 131, 3), 31)
    plan = _compiled(flat, cuda_device)
    assert plan.handle.rows_need_padding()
    s = _assert_counts(plan, classify(flat))
    assert s["fast"] > 0
    assert compare_u8(_run(plan, src, cuda_device).cpu().numpy(), _warp_ref(src, flat)) == (0, 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("channels", [1, 4])
def test_other_channel_counts_have_no_fast_tiles(cuda_device, channels):
    shape = PHASE_SRC if channels == 1 else PHASE_SRC + (channels,)
    src = _noise(shape, 32)
    for i, j in PHASES:
        flat = single_layer(phase_A(i, j), PHASE_SRC, 256, 64, channels)
        plan = _compiled(flat, cuda_device)
        s = plan.handle.tiled_stats()
        assert s["fast"] == 0 and s["warp"] == 8, s
        assert compare_u8(_run(plan, src, cuda_device).cpu().numpy(), _warp_ref(src, flat)) == (0, 1.0), (i, j)


@pytest.mark.gpu
def test_window_uploads_on_a_translation_rig(cuda_device):
    """The group window reads five words from its anchor: with the device slots poisoned outside the uploaded
    windows, no byte of the poison may reach the panorama."""
    import torch
    from multicamera_stitching_b200 import Stitcher
    from multicamera_stitching_b200.sequence import SequencePipeline, pinned_like
    h, w = 120, 320
    steps = [(200.37, 3.71), (150.84, -4.29)]
    states = translation_chain(3, h, w, steps, 5, 6)
    labels = ["CAM1", "CAM2", "CAM3"]
    images = {l: _noise((h, w, 3), 40 + k) for k, l in enumerate(labels)}
    st = Stitcher(images)
    shapeB = (h, w, 3)
    for k, step in enumerate(steps):
        st.stitchers[k].set_homography(A_translate(*step), (h, w, 3), shapeB, 5, 6)
        shapeB = st.stitchers[k].result_shape()
    shapes = [(h, w, 3)] * 3
    F = 5
    sets = [{l: _noise((h, w, 3), 100 * f + k) for k, l in enumerate(labels)} for f in range(F)]
    host = {l: pinned_like((F, h, w, 3)) for l in labels}
    for l in labels:
        for f in range(F):
            host[l][f].copy_(torch.from_numpy(sets[f][l]))
    pipe = SequencePipeline(st, shapes, cuda_device, chunk=2, depth=2)
    s = pipe.plan.handle.tiled_stats()
    assert s["fast"] > 0, s
    assert pipe.bytes_per_frame()[0] < 3 * h * w * 3
    for slot in pipe.slots:
        for t in slot["src"]:
            t.fill_(0xAB)
    out = pinned_like((F,) + pipe.plan.out_shape())
    assert pipe.run(host, out) == F
    assert pipe.plan.handle.last_variant() == 2
    for f in range(F):
        assert compare_u8(out[f].numpy(), stitcher_ref.stitch_chain(states, labels, sets[f])) == (0, 1.0), f


# ---- CPU: the chosen geometries stay on the path ---------------------------------------------------------------------
def test_model_geometries_select_fast_tiles():
    for i, j in PHASES:
        m = classify(single_layer(phase_A(i, j), PHASE_SRC, 256, 64))
        assert (m["fast"], m["warp"], m["fast_passes"]) == (8, 0, 0), (i, j, m)
    for name, A in GENERAL.items():
        m = classify(single_layer(A, (360, 640), 640, 360))
        assert m["fast"] > 0 and m["fast_passes"] == 1, (name, m)
        assert max(m["max_off"]) > 0
        if name in ("scale1.02", "scale1.04"):
            assert m["warp"] > 0, (name, m)
        if name == "scale1.005":
            assert m["warp"] == 0 and max(m["max_off"]) > 6
    m = classify(single_layer(GENERAL["scale1.04"], (360, 640), 640, 360), limit=64)
    assert m["fast_passes"] == 2
    for name in GENERAL:
        m0 = classify(single_layer(GENERAL[name], (360, 640), 640, 360), limit=0)
        assert m0["fast"] == sum(v == 0 for v in m0["max_off"])
    mixed = False
    for src_hw, out_wh, tx, ty in BORDERS:
        flat = single_layer(A_translate(tx, ty), src_hw, *out_wh)
        assert all(_clamped_sides(flat)), (tx, ty)
        m = classify(flat)
        assert m["fast"] > 0, (tx, ty, m)
        mixed |= m["warp"] > 0 and m["fast_passes"] == 0
        if m["warp"] == 0:
            assert m["fast_passes"] == 1     # the clamped columns are on the general lists
    assert mixed
    for xoffset in (1, 2, 3):
        flat = chain_flat(translation_chain(2, 120, 640, [ANCHOR_STEP], xoffset, 4), 120, 640)
        assert flat.layers[0].rect[2] % 4 == xoffset
        assert _unanchored(flat) > 0
        assert classify(flat)["fast"] > 0
    m = classify(single_layer(A_translate(3.37, 2.59), (80, 131), 128, 64))
    assert m["fast"] > 0
    for w in (253, 256):
        m = classify(single_layer(phase_A(13, 11), PHASE_SRC, w, 64))
        assert m["fast"] > 0 and m["warp"] == 0
    m = classify(single_layer(phase_A(7, 17), PHASE_SRC, 256, 64), pitch_words=4)
    assert m["fast"] == 8
