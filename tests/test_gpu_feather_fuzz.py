"""Fused seam blend on the GPU, fuzzed: the BAND-aware tiled kernel (``mcs_stitch_tiled_kernel<C, true>``, the
multi-box issuer), the plan-time ``mcs_band_bounds_kernel`` / ``mcs_band_desc_kernel`` and the overlay windows the
host uploads, bit for bit against ``oracle/feather_model.py``.

a. the seeded random rigs (rotated, mirrored, perspective cameras; super-mode crops trimmed so that they cut pasted
   rectangles) under the ramp and weight maps of every kind, numpy frames and device batches; plans the fused form
   cannot express (more than two outer layers in one tile) take the two-pass form or refuse their maps;
b. frame counts on both sides of the launcher's split rule (restated in ``feather_cases.split_rule``): BAND tiles cut
   into frame chunks, last frame blocks too short to split, frame blocks of 16 and 4, FAST and BAND tiles in one
   split launch;
c. output layouts: odd bases, padded pitches, frame strides that move the 16-byte phase, into poisoned buffers;
d. source layouts the engine realigns (scratch copy, zero-padded rows), an unaligned source through the C ABI
   (gather + two-pass band kernel, or the refusal of a plan with maps), forced variants;
e. weight maps at their extremes (0, 1, F - 1, F, above F, checkerboards, masks) handed over as windows of wider
   arrays through ``mcs_plan_set_blend``;
f. everything outside the source windows poisoned, in frames, staging tensors and pipeline slots."""
import ctypes
import os

import numpy as np
import pytest

import feather_cases as fc
from helpers import synthetic_chain
from multicamera_stitching_b200 import _cabi
from multicamera_stitching_b200.plan import plan_paste
from oracle import feather_model, stitcher_ref
from random_rigs import mirrored

pytestmark = pytest.mark.gpu

SEEDS = range(28)
FUSED_ERROR = "fused band form"

# what the file exercised, asserted by the last test
COVERED = {"log2": set(), "channels": set(), "mirrored": set(), "cut": set(), "two_overlays": set(),
           "zero_base": set(), "kinds": set(), "band_split": set(), "dropped": set(), "fast_band_split": 0,
           "moving_phase": 0, "variant3_from_fused": 0, "unfused": set(), "hidden": set(), "channels_split": set()}


def _rig(seed):
    made = fc.rig(seed)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    return made


def _channels(images, labels):
    a = images[labels[0]]
    return 1 if a.ndim == 2 else a.shape[2]


def _frames(images, labels, rng):
    return {l: rng.integers(0, 256, size=images[l].shape, dtype=np.uint8) for l in labels}


def _batch(torch, sets, labels, device):
    return {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(device) for l in labels}


def _diff(got, ref):
    return int(np.abs(got.astype(int) - ref.astype(int)).max()) if got.shape == ref.shape else (got.shape, ref.shape)


def _fresh(st):
    """Drop the stitcher's plan cache (the $MCS_TILED_* switches are read when a plan is built)."""
    st.__dict__.pop("_engine", None)


def _record_tiles(seed, tiles):
    if any(n == 2 for n, _ in tiles):
        COVERED["two_overlays"].add(seed)
    if any(z for _, z in tiles):
        COVERED["zero_base"].add(seed)


# ---- a. random rigs -------------------------------------------------------------------------------------------------

A_KINDS = ("random", "zero", "one", "fm1", "full", "over", "checker")


@pytest.mark.parametrize("seed", SEEDS)
def test_random_rig_matches_the_specification(cuda_device, seed):
    import torch
    st, states, labels, images = _rig(seed)
    flat = fc.plan_flat(st, images, labels)
    shapes = [images[l].shape for l in labels]
    log2 = 1 + seed % 5
    cut = fc.is_cut(flat)
    rng = np.random.default_rng(500 + seed)
    sets = [_frames(images, labels, rng) for _ in range(3)]
    batch = _batch(torch, sets, labels, cuda_device)

    # the distance ramp
    tiles = fc.band_tiles(flat, log2)
    fused = max([n for n, _ in tiles], default=0) <= fc.MAX_OVERLAYS
    st.feather_log2 = log2
    ref = feather_model.feather_chain(states, labels, images, log2)
    if cut and not fused:
        with pytest.raises(_cabi.McsError, match=FUSED_ERROR):
            st.stitch(images)
    else:
        got = st.stitch(images)
        assert got.shape == ref.shape and np.array_equal(got, ref), _diff(got, ref)
        plan = st.plan(shapes, cuda_device)
        s = plan.handle.tiled_stats()
        assert s["band_fused"] == int(fused), (s, tiles)
        assert plan.handle.last_variant() == (4 if fused else 3)
        if fused:
            assert s["band"] == len(tiles), (s, len(tiles))
            _record_tiles(seed, tiles)
        else:
            COVERED["unfused"].add(seed)
        out = st.stitch_batch(batch).cpu().numpy()
        for f, fr in enumerate(sets):
            assert np.array_equal(out[f], feather_model.feather_chain(states, labels, fr, log2)), f

    # weight maps
    kind = A_KINDS[seed % len(A_KINDS)]
    maps = fc.make_maps(fc.stage_shapes(st, images, labels), log2, kind, seed=seed)
    tiles = fc.band_tiles(flat, log2, maps)
    st.blend_weights = maps
    if max([n for n, _ in tiles], default=0) > fc.MAX_OVERLAYS:
        with pytest.raises(_cabi.McsError, match=FUSED_ERROR):
            st.stitch(images)
        COVERED["unfused"].add(seed)
        return
    ref = feather_model.feather_chain(states, labels, images, log2, maps)
    got = st.stitch(images)
    assert got.shape == ref.shape and np.array_equal(got, ref), _diff(got, ref)
    if kind == "full":
        assert np.array_equal(got, stitcher_ref.stitch_chain(states, labels, images))
    plan = st.plan(shapes, cuda_device)
    s = plan.handle.tiled_stats()
    assert s["band_fused"] == 1 and s["band"] == len(tiles) and plan.handle.last_variant() == 4, (s, len(tiles))
    out = st.stitch_batch(batch).cpu().numpy()
    for f, fr in enumerate(sets):
        assert np.array_equal(out[f], feather_model.feather_chain(states, labels, fr, log2, maps)), f
    _record_tiles(seed, tiles)
    COVERED["log2"].add(log2)
    COVERED["channels"].add(_channels(images, labels))
    COVERED["kinds"].add(kind)
    if mirrored(seed):
        COVERED["mirrored"].add(seed)
    if cut:
        COVERED["cut"].add(seed)


# ---- b. frame counts and the split ----------------------------------------------------------------------------------

PERIOD = 7   # distinct frame-sets of a long batch: no frame block (64, 16, 4) or chunk (16, 4, 1 frames) is a multiple
FRAME_COUNTS = (1, 3, 15, 16, 17, 64, 65, 67, 68, 80, 130)


def _split_rig(name):
    """Rigs with many BAND tiles: ``(stitcher, states, labels, images, feather_log2, maps or None)``."""
    if name == "synthetic6":
        st, states, labels, images = synthetic_chain(6, 270, 480, 3, kind="noise", xoffset=2, yoffset=7)
        return st, states, labels, images, 3, None
    seed, log2, kind = {"rig9": (9, 3, None), "rig25": (25, 4, "random"), "rig24": (24, 5, None)}[name]
    st, states, labels, images = _rig(seed)
    maps = None if kind is None else fc.make_maps(fc.stage_shapes(st, images, labels), log2, kind, seed=seed)
    return st, states, labels, images, log2, maps


def _split_of(plan, n_frames):
    import torch
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    per_sm = plan.handle.tiled_ctas_per_sm()
    assert per_sm >= 1
    s = plan.handle.tiled_stats()
    return s, fc.split_rule(s, per_sm, n_sm, n_frames)


def _long_batch(torch, st, states, labels, images, log2, maps, device, seed):
    rng = np.random.default_rng(seed)
    sets = [_frames(images, labels, rng) for _ in range(PERIOD)]
    refs = [feather_model.feather_chain(states, labels, fr, log2, maps) for fr in sets]
    distinct = _batch(torch, sets, labels, device)
    return refs, distinct


def _run_counts(torch, st, labels, distinct, refs, counts, shapes, device, tag):
    """Stitch batches of ``counts`` frames (frame f = distinct set f % PERIOD); returns the split of each launch."""
    seen = {}
    for F in counts:
        idx = torch.arange(F, device=device) % PERIOD
        batch = {l: distinct[l][idx].contiguous() for l in labels}
        out = st.stitch_batch(batch).cpu().numpy()
        plan = st.plan(shapes, device)
        assert plan.handle.last_variant() == 4
        for f in range(F):
            assert np.array_equal(out[f], refs[f % PERIOD]), (tag, F, f)
        s, (split, first, end) = _split_of(plan, F)
        assert s["band"] > 0
        fb = min(s["frame_block"], F)
        nf_last = F - (-(-F // fb) - 1) * fb
        want_split = os.environ.get("MCS_TILED_SPLIT")
        want = (int(want_split) if want_split else (4 if fb >= 16 else 1))
        if want > 1 and nf_last >= want:
            # the split really cuts BAND tiles (they come first in the table)
            assert split == want and first < s["band"], (tag, F, s, split, first, end)
            COVERED["band_split"].add((tag, F))
        else:
            assert split == 1, (tag, F, split)
            if want > 1:
                COVERED["dropped"].add(F)
        seen[F] = (split, first, end, s)
    return seen


@pytest.mark.parametrize("name", ["synthetic6", "rig9", "rig25", "rig24"])
def test_frame_counts_split_band_tiles(cuda_device, name):
    import torch
    st, states, labels, images, log2, maps = _split_rig(name)
    st.feather_log2, st.blend_weights = log2, maps
    shapes = [images[l].shape for l in labels]
    refs, distinct = _long_batch(torch, st, states, labels, images, log2, maps, cuda_device, 77)
    _run_counts(torch, st, labels, distinct, refs, FRAME_COUNTS, shapes, cuda_device, name)
    COVERED["channels_split"].add(_channels(images, labels))


@pytest.mark.parametrize("block,split,counts", [(16, None, (20, 33)), (4, "4", (12, 11, 1, 5))])
def test_split_with_other_frame_blocks(cuda_device, monkeypatch, block, split, counts):
    """A frame block of 16 whose last block holds 4 frames (split in four), and blocks of 4 frames cut into chunks of
    one frame by $MCS_TILED_SPLIT=4 (dropped where the last block is shorter)."""
    import torch
    st, states, labels, images, log2, maps = _split_rig("rig9")
    monkeypatch.setenv("MCS_TILED_FRAME_BLOCK", str(block))
    if split:
        monkeypatch.setenv("MCS_TILED_SPLIT", split)
    _fresh(st)
    st.feather_log2 = log2
    shapes = [images[l].shape for l in labels]
    refs, distinct = _long_batch(torch, st, states, labels, images, log2, None, cuda_device, 78)
    seen = _run_counts(torch, st, labels, distinct, refs, counts, shapes, cuda_device, "block%d" % block)
    assert seen[counts[0]][0] == 4
    assert st.plan(shapes, cuda_device).handle.tiled_stats()["frame_block"] == block


def test_split_launch_with_fast_and_band_tiles(cuda_device):
    """A translation rig (test_gpu_fast_tiles.py): FAST and BAND tiles in one launch, both cut into frame chunks."""
    import torch
    from multicamera_stitching_b200 import Stitcher
    from test_gpu_fast_tiles import A_translate, translation_chain
    h, w, log2 = 96, 320, 3
    steps = [(200.37, 3.71), (150.84, -4.29)]
    states = translation_chain(3, h, w, steps, 5, 6)
    labels = ["CAM1", "CAM2", "CAM3"]
    images = {l: np.random.default_rng(40 + k).integers(0, 256, size=(h, w, 3), dtype=np.uint8)
              for k, l in enumerate(labels)}
    st = Stitcher(images)
    shapeB = (h, w, 3)
    for k, step in enumerate(steps):
        st.stitchers[k].set_homography(A_translate(*step), (h, w, 3), shapeB, 5, 6)
        shapeB = st.stitchers[k].result_shape()
    st.feather_log2 = log2
    shapes = [(h, w, 3)] * 3
    refs, distinct = _long_batch(torch, st, states, labels, images, log2, None, cuda_device, 79)
    seen = _run_counts(torch, st, labels, distinct, refs, (16, 64, 65), shapes, cuda_device, "translation")
    split, first, end, s = seen[64]
    assert s["fast"] > 0 and s["band"] > 0 and split == 4
    assert first < s["band"] and end == s["band"] + s["fast"] + s["warp"]   # BAND and FAST tiles among the cut ones
    COVERED["fast_band_split"] += 1


# ---- c. output layouts ----------------------------------------------------------------------------------------------

# (seed, base offset, row pad, frame-stride pad, frames, weight maps)
OUT_LAYOUTS = [(9, 0, 1, 0, 3, False), (5, 1, 7, 5, 4, True), (25, 2, 16, 3, 5, True), (14, 3, 64, 0, 2, False),
               (20, 4, 1, 13, 17, False), (12, 5, 7, 1, 3, True), (6, 0, 16, 7, 16, True), (16, 3, 64, 2, 1, True),
               (13, 1, 16, 9, 6, True), (2, 0, 64, 4, 5, True)]


def _setup(st, images, labels, seed, log2, with_maps):
    maps = fc.make_maps(fc.stage_shapes(st, images, labels), log2, "random", seed=seed) if with_maps else None
    st.feather_log2, st.blend_weights = log2, maps
    return maps


def _dense_frames(torch, sets, labels, device):
    return [torch.from_numpy(np.stack([s[l] for s in sets])).to(device) for l in labels]


@pytest.mark.parametrize("seed,offset,row_pad,fpad,F,with_maps", OUT_LAYOUTS)
def test_output_layouts_into_a_poisoned_buffer(cuda_device, seed, offset, row_pad, fpad, F, with_maps):
    import torch
    st, states, labels, images = _rig(seed)
    log2 = 1 + (seed + 2) % 5
    maps = _setup(st, images, labels, seed, log2, with_maps)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.tiled_stats()["band_fused"] == 1 and plan.handle.tiled_stats()["band"] > 0
    rng = np.random.default_rng(900 + seed)
    sets = [_frames(images, labels, rng) for _ in range(F)]
    C = plan.channels
    row = plan.out_w * C
    pitch = row + row_pad
    fstride = plan.out_h * pitch + fpad
    total = offset + F * fstride + 64
    poison = torch.full((total,), 0xAB, dtype=torch.uint8, device=cuda_device)
    shape = (F, plan.out_h, plan.out_w) + ((C,) if plan.flat.ndim == 3 else ())
    strides = (fstride, pitch) + ((C, 1) if plan.flat.ndim == 3 else (1,))
    out = torch.as_strided(poison, shape, strides, offset)
    plan.run(_dense_frames(torch, sets, labels, cuda_device), out=out, n_frames=F)
    assert plan.handle.last_variant() == 4
    got = out.cpu().numpy()
    for f in range(F):
        assert np.array_equal(got[f], feather_model.feather_chain(states, labels, sets[f], log2, maps)), f
    written = np.zeros(total, bool)
    written[np.lib.stride_tricks.as_strided(np.arange(offset, total), shape, [s * 8 for s in strides]).ravel()] = True
    assert bool((poison.cpu().numpy()[~written] == 0xAB).all())
    phases = {(offset + f * fstride + y * pitch) % 16 for f in range(F) for y in range(plan.out_h)}
    if len(phases) > 1:
        COVERED["moving_phase"] += 1


# ---- d. source layouts, the C ABI's fallbacks, forced variants ------------------------------------------------------

def _strided_sources(torch, rng, sets, labels, images, layout, device):
    """Device views of ``sets`` with base offsets / pitches / frame strides of ``layout``; returns the views and
    whether any of them is off the 16-byte grid the tiled kernel takes."""
    F = len(sets)
    views, odd = [], False
    odd_cam = int(rng.integers(0, len(labels)))
    for k, l in enumerate(labels):
        shp = images[l].shape
        h, w = shp[:2]
        C = 1 if len(shp) == 2 else shp[2]
        row = w * C
        off, pitch, fpad = 0, row + (-row) % 16, 0
        if k == odd_cam or layout == "odd_base":
            if layout == "odd_base":
                off = int(rng.integers(1, 16))
            elif layout == "odd_pitch":
                pitch = row + int(rng.integers(1, 16)) | 1
            elif layout == "odd_fstride":
                fpad = int(rng.integers(1, 16)) | 1
        fstride = h * pitch + fpad
        buf = torch.full((off + F * fstride + 16,), 0x5A, dtype=torch.uint8, device=device)
        shape, strides = ((F, h, w, C), (fstride, pitch, C, 1)) if len(shp) == 3 else ((F, h, w), (fstride, pitch, 1))
        v = torch.as_strided(buf, shape, strides, off)
        v.copy_(torch.from_numpy(np.stack([s[l] for s in sets])).to(device))
        odd = odd or (v.data_ptr() % 16 != 0 or pitch % 16 != 0 or (F > 1 and fstride % 16 != 0))
        views.append(v)
    return views, odd


# rows of 65 (seed 4, C = 1), 129 (9, C = 1), 633 (14, C = 3), 146 (19, C = 1) and 339 bytes (24, C = 3): none a
# multiple of 4, so the engine passes them through zero-padded scratch rows (mcs_plan_promise_padded_rows)
SRC_LAYOUTS = [(1, "odd_base", 3), (6, "odd_pitch", 2), (13, "odd_fstride", 4), (25, "odd_base", 1),
               (17, "odd_pitch", 5), (3, "odd_fstride", 3), (4, "padded_rows", 3), (9, "padded_rows", 1),
               (14, "padded_rows", 2), (19, "padded_rows", 4), (24, "padded_rows", 2)]


@pytest.mark.parametrize("seed,layout,F", SRC_LAYOUTS)
def test_source_layouts_the_engine_realigns(cuda_device, seed, layout, F):
    import torch
    st, states, labels, images = _rig(seed)
    log2 = 1 + (seed + 3) % 5
    flat = fc.plan_flat(st, images, labels)
    maps = fc.make_maps(fc.stage_shapes(st, images, labels), log2, "random", seed=seed)
    if max([n for n, _ in fc.band_tiles(flat, log2, maps)], default=0) > fc.MAX_OVERLAYS:
        maps = None
    st.feather_log2, st.blend_weights = log2, maps
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.tiled_stats()["band_fused"] == 1
    assert plan.handle.rows_need_padding() == (layout == "padded_rows")
    rng = np.random.default_rng(1200 + seed)
    sets = [_frames(images, labels, rng) for _ in range(F)]
    views, odd = _strided_sources(torch, rng, sets, labels, images, layout, cuda_device)
    assert odd == (layout != "padded_rows" and (layout != "odd_fstride" or F > 1))
    got = plan.run(views, n_frames=F).cpu().numpy()
    assert plan.handle.last_variant() == 4
    for f in range(F):
        assert np.array_equal(got[f], feather_model.feather_chain(states, labels, sets[f], log2, maps)), f


def _direct(plan, views, F, out):
    """``mcs_stitch_u8`` straight through the C ABI, with the sources as they are (no realignment)."""
    ptrs = [v.data_ptr() for v in views]
    pitches = [v.stride()[1] for v in views]
    fstrides = [v.stride()[0] for v in views]
    plan.handle.stitch(ptrs, pitches, fstrides, F, out.data_ptr(), out.stride()[1], out.stride()[0])


@pytest.mark.parametrize("seed", [0, 5, 10, 13, 25])
def test_fallbacks_of_a_fused_plan(cuda_device, seed):
    """A fused plan served by the gather kernel (an unaligned source through the C ABI, or variant 1 forced) blends
    its bands in the two-pass form (variant 3); with weight maps it cannot, refuses the call and stays usable."""
    import torch
    st, states, labels, images = _rig(seed)
    flat = fc.plan_flat(st, images, labels)
    assert not fc.is_cut(flat)
    log2 = 1 + seed % 5
    F = 3
    rng = np.random.default_rng(1300 + seed)
    sets = [_frames(images, labels, rng) for _ in range(F)]
    views, odd = _strided_sources(torch, rng, sets, labels, images, "odd_base", cuda_device)
    assert odd
    dense = _dense_frames(torch, sets, labels, cuda_device)

    st.feather_log2, st.blend_weights = log2, None
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.tiled_stats()["band_fused"] == 1
    refs = [feather_model.feather_chain(states, labels, s, log2) for s in sets]
    out = plan.new_output(F)
    _direct(plan, views, F, out)
    assert plan.handle.last_variant() == 3
    for f in range(F):
        assert np.array_equal(out[f].cpu().numpy(), refs[f]), f
    for variant, want in ((1, 3), (2, 4), (0, 4)):
        plan.handle.force_variant(variant)
        try:
            got = plan.run(dense, n_frames=F).cpu().numpy()
            assert plan.handle.last_variant() == want, variant
        finally:
            plan.handle.force_variant(0)
        for f in range(F):
            assert np.array_equal(got[f], refs[f]), (variant, f)
    COVERED["variant3_from_fused"] += 1

    maps = fc.make_maps(fc.stage_shapes(st, images, labels), log2, "checker", seed=seed)
    if max([n for n, _ in fc.band_tiles(flat, log2, maps)], default=0) > fc.MAX_OVERLAYS:
        return
    st.blend_weights = maps
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    refs = [feather_model.feather_chain(states, labels, s, log2, maps) for s in sets]
    out = plan.new_output(F)
    with pytest.raises(_cabi.McsError, match="code -3"):
        _direct(plan, views, F, out)
    plan.handle.force_variant(1)
    try:
        with pytest.raises(_cabi.McsError, match="code -3"):
            plan.run(dense, n_frames=F)
    finally:
        plan.handle.force_variant(0)
    got = plan.run(views, n_frames=F).cpu().numpy()   # the engine realigns: the fused form again
    assert plan.handle.last_variant() == 4
    for f in range(F):
        assert np.array_equal(got[f], refs[f]), f


# ---- e. weights at their extremes, through the C ABI ----------------------------------------------------------------

E_KINDS = ("zero", "one", "fm1", "full", "over", "checker")
E_SEEDS = (0, 2, 4, 6, 9, 11, 13, 15, 19, 25, 27)   # rigs whose every map kind fits the fused form


def _set_blend_windows(plan, log2, maps):
    """``mcs_plan_set_blend`` with every map handed over as the left part of a wider array (map_pitch > width)
    whose padding would change the panorama if it were read.  Returns the return code."""
    lmaps = fc.layer_maps(plan.flat, maps)
    n = len(lmaps)
    ptrs = (ctypes.c_void_p * n)()
    pitches = np.zeros(n, np.int64)
    keep = []
    for k, m in enumerate(lmaps):
        if m is None:
            continue
        h, w = m.shape
        big = np.full((h, w + 1 + 6 * k), 0 if m.max() > 0 else 255, np.uint8)
        big[:, :w] = m
        keep.append(big)
        ptrs[k] = big.ctypes.data
        pitches[k] = big.strides[0]
    paste = np.ascontiguousarray(plan_paste(plan.flat), dtype=np.int32)
    lib = _cabi.load()
    return lib.mcs_plan_set_blend(plan.handle._h, int(log2), paste.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                  ptrs, pitches.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))


@pytest.mark.parametrize("log2", [0, 1, 4, 5])
@pytest.mark.parametrize("kind", E_KINDS + ("mask",))
def test_weight_extremes_through_the_c_abi(cuda_device, kind, log2):
    import torch
    from multicamera_stitching_b200.engine import CompiledPlan
    if kind == "mask" and log2 != 0:
        pytest.skip("0 / 1 masks are the weights of feather_log2 = 0")
    seed = E_SEEDS[(3 * (E_KINDS + ("mask",)).index(kind) + log2) % len(E_SEEDS)]
    st, states, labels, images = _rig(seed)
    flat = fc.plan_flat(st, images, labels)
    maps = fc.make_maps(fc.stage_shapes(st, images, labels), log2, kind, seed=seed + log2)
    tiles = fc.band_tiles(flat, log2, maps)
    assert max([n for n, _ in tiles], default=0) <= fc.MAX_OVERLAYS
    plan = CompiledPlan(flat, cuda_device)
    rc = _set_blend_windows(plan, log2, maps)
    assert rc == 0, _cabi.load().mcs_last_error().decode()
    if plan.handle.rows_need_padding():
        plan.pad_rows = True
        plan.handle.promise_padded_rows(True)
    rng = np.random.default_rng(1400 + seed)
    sets = [_frames(images, labels, rng) for _ in range(2)]
    got = plan.run(_dense_frames(torch, sets, labels, cuda_device), n_frames=2).cpu().numpy()
    assert plan.handle.last_variant() == 4
    s = plan.handle.tiled_stats()
    assert s["band_fused"] == 1 and s["band"] == len(tiles), (s, len(tiles))
    F = 1 << log2
    for f, fr in enumerate(sets):
        ref = feather_model.feather_chain(states, labels, fr, log2, maps)
        assert np.array_equal(got[f], ref), (f, _diff(got[f], ref))
        if kind == "full":
            assert np.array_equal(ref, stitcher_ref.stitch_chain(states, labels, fr))
        if kind == "over":
            clipped = [np.minimum(m, F).astype(np.uint8) for m in maps]
            assert np.array_equal(ref, feather_model.feather_chain(states, labels, fr, log2, clipped))
    _record_tiles(seed, tiles)
    COVERED["kinds"].add(kind)
    COVERED["log2"].add(log2)


def test_weight_maps_beyond_five_feather_bits_are_refused(cuda_device):
    from multicamera_stitching_b200.engine import CompiledPlan
    st, states, labels, images = _rig(2)
    flat = fc.plan_flat(st, images, labels)
    maps = fc.make_maps(fc.stage_shapes(st, images, labels), 6, "random", seed=2)
    plan = CompiledPlan(flat, cuda_device)
    assert _set_blend_windows(plan, 6, maps) == -1
    assert "feather_log2 <= 5" in _cabi.load().mcs_last_error().decode()
    st.feather_log2, st.blend_weights = 6, maps
    with pytest.raises(_cabi.McsError, match="code -1"):
        st.stitch(images)
    # the refused plan is still the overwrite
    import torch
    got = plan.run(_dense_frames(torch, [images], labels, cuda_device), n_frames=1).cpu().numpy()[0]
    assert np.array_equal(got, stitcher_ref.stitch_chain(states, labels, images))


# ---- f. source windows: everything else poisoned ----------------------------------------------------------------------

def _poison_outside_spans(plan, images, labels, rows):
    """Frames with every byte outside the plan's per-band source spans (``rows`` source rows a band) inverted."""
    C = plan.channels
    out = {}
    for k, l in enumerate(labels):
        h = images[l].shape[0]
        row = images[l].size // h
        keep = np.zeros((h, row), bool)
        for b, (x0, x1) in enumerate(plan.handle.source_spans(k, rows)):
            if x1 > x0:
                keep[b * rows:(b + 1) * rows, max(0, x0) * C:x1 * C] = True
        flat = images[l].reshape(h, row).copy()
        flat[~keep] = 255 - flat[~keep]
        out[l] = flat.reshape(images[l].shape)
    return out


@pytest.mark.parametrize("seed", SEEDS)
def test_source_windows_on_random_rigs(cuda_device, seed):
    import torch
    st, states, labels, images = _rig(seed)
    flat = fc.plan_flat(st, images, labels)
    log2 = 1 + (seed + 1) % 5
    maps = fc.make_maps(fc.stage_shapes(st, images, labels), log2, "random", seed=seed + 7)
    if max([n for n, _ in fc.band_tiles(flat, log2, maps)], default=0) > fc.MAX_OVERLAYS:
        maps = None
    st.feather_log2, st.blend_weights = log2, maps
    ref = feather_model.feather_chain(states, labels, images, log2, maps)
    assert np.array_equal(st.stitch(images), ref)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.last_variant() == 4
    # device frames poisoned outside the exact spans of every source row
    tight = _poison_outside_spans(plan, images, labels, 1)
    if any(not np.array_equal(tight[l], images[l]) for l in labels):
        COVERED["hidden"].add(seed)   # elsewhere every source row is read over its whole width
    got = st.stitch_batch({l: torch.from_numpy(tight[l][None]).to(cuda_device) for l in labels})[0].cpu().numpy()
    assert np.array_equal(got, ref), _diff(got, ref)
    # numpy frames poisoned outside upload_bands(), and the staging tensors outside the windows they receive
    bands = plan.upload_bands()
    poisoned = {}
    for k, l in enumerate(labels):
        row, rows, copies = bands[k]
        keep = np.zeros((rows, row), bool)
        for cp in copies:
            keep[cp["y0"]:cp["y0"] + cp["rows"], cp["b0"]:cp["b0"] + cp["nbytes"]] = True
        fl = images[l].reshape(rows, row).copy()
        fl[~keep] = 255 - fl[~keep]
        poisoned[l] = fl.reshape(images[l].shape)
    for t in st._engine_()._staging.values():
        t.fill_(0x5A)
    got = st.stitch(poisoned)
    assert np.array_equal(got, ref), _diff(got, ref)


def test_sequence_pipeline_with_poisoned_slots(cuda_device):
    import torch
    from multicamera_stitching_b200.sequence import SequencePipeline, pinned_like
    st, states, labels, images = _rig(24)
    log2 = 5
    st.feather_log2 = log2
    shapes = [images[l].shape for l in labels]
    pipe = SequencePipeline(st, shapes, cuda_device, chunk=3, depth=2)
    assert 0 < pipe.bytes_per_frame()[0] < sum(int(np.prod(s)) for s in shapes)
    assert pipe.plan.handle.tiled_stats()["band_fused"] == 1
    F = 7
    rng = np.random.default_rng(24)
    sets = [_frames(images, labels, rng) for _ in range(F)]
    host = {l: torch.from_numpy(np.stack([s[l] for s in sets])).pin_memory() for l in labels}
    for slot in pipe.slots:
        for t in slot["src"]:
            t.fill_(0xA5)
    out = pinned_like((F,) + pipe.plan.out_shape())
    assert pipe.run(host, out) == F
    assert pipe.plan.handle.last_variant() == 4
    for f in range(F):
        assert np.array_equal(out[f].numpy(), feather_model.feather_chain(states, labels, sets[f], log2)), f


# ---- h. what the file exercised --------------------------------------------------------------------------------------

def test_fuzz_exercised_the_fused_blend(cuda_device):
    assert COVERED["band_split"], COVERED
    assert {65, 67, 130} <= COVERED["dropped"], COVERED
    assert COVERED["fast_band_split"] >= 1, COVERED
    assert COVERED["two_overlays"] and COVERED["zero_base"], COVERED
    assert COVERED["channels"] >= {1, 3, 4} and COVERED["channels_split"] >= {1, 3, 4}, COVERED
    assert COVERED["log2"] >= {0, 1, 2, 3, 4, 5}, COVERED
    assert COVERED["kinds"] >= set(A_KINDS) | {"mask"}, COVERED
    assert COVERED["mirrored"] and COVERED["cut"], COVERED
    assert COVERED["moving_phase"] >= 1, COVERED
    assert COVERED["variant3_from_fused"] >= 1, COVERED
    assert COVERED["unfused"], COVERED
    assert len(COVERED["hidden"]) >= 5, COVERED
