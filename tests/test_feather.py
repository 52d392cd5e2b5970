"""Feather blend mode (SURVEY.md section 8 row f1, an extension the reference does not have):
the numpy specification reduces to the reference's overwrite, and the CUDA kernel matches the
specification bit for bit."""
import cv2
import numpy as np
import pytest

from helpers import synthetic_chain
from oracle import feather_model, stitcher_ref


@pytest.mark.parametrize("n,h,w,c", [(2, 64, 96, 3), (3, 120, 200, 3), (4, 90, 160, 1)])
def test_feather_width_one_is_the_reference_overwrite(n, h, w, c):
    st, states, labels, images = synthetic_chain(n, h, w, c, kind="noise", xoffset=3, yoffset=5)
    assert np.array_equal(feather_model.feather_chain(states, labels, images, 0),
                          stitcher_ref.stitch_chain(states, labels, images))


def test_feather_only_touches_the_seam_band():
    st, states, labels, images = synthetic_chain(3, 120, 200, 3, kind="noise")
    hard = stitcher_ref.stitch_chain(states, labels, images)
    soft = feather_model.feather_chain(states, labels, images, 3)
    assert soft.shape == hard.shape
    changed = (soft != hard).any(axis=2)
    assert changed.any()
    # camera 0 keeps its pixels further than 8 px (+ one stage of nesting) from its border
    bx = sum(int(s["Bpts"][0][0]) for s in states)
    by = sum(int(s["Bpts"][0][1]) for s in states)
    h, w = images[labels[0]].shape[:2]
    assert not changed[by + 8:by + h - 8, bx + 8:bx + w - 8].any()


def _random_weights(states, images, labels, log2, seed=0):
    """One weight map per stage (shape of that stage's imageB = the running canvas), values 0 .. F with
    plateaus of F (most of a real map is 'keep the canvas')."""
    rng = np.random.default_rng(seed)
    F = 1 << log2
    maps = []
    shapeB = images[labels[0]].shape[:2]
    for st in states:
        m = rng.integers(0, F + 1, size=shapeB, dtype=np.int64)
        keep = rng.random(shapeB) < 0.5
        m[keep] = F
        maps.append(m.astype(np.uint8))
        dst = stitcher_ref.stitch_pair(st, (np.zeros(shapeB + images[labels[0]].shape[2:], np.uint8),
                                            np.zeros(st["AimgSize"], np.uint8)))
        shapeB = dst.shape[:2]
    return maps


def test_weight_maps_generalise_the_ramp_and_reduce_to_the_overwrite():
    st, states, labels, images = synthetic_chain(3, 120, 200, 3, kind="noise")
    hard = stitcher_ref.stitch_chain(states, labels, images)
    # the ramp as explicit maps
    shapes_b = [m.shape for m in _random_weights(states, images, labels, 3)]
    ramps = [feather_model.ramp_weights(sh, 3) for sh in shapes_b]
    assert np.array_equal(feather_model.feather_chain(states, labels, images, 3, ramps),
                          feather_model.feather_chain(states, labels, images, 3))
    # full weight everywhere = the reference's overwrite (StitcherClass.py:240-241), at any F
    for log2 in (0, 3):
        full = [np.full(sh, 1 << log2, np.uint8) for sh in shapes_b]
        assert np.array_equal(feather_model.feather_chain(states, labels, images, log2, full), hard)
    # F = 1 and a {0, 1} mask: 0 shows the warped camera where it touches its source
    mask = [np.ones(sh, np.uint8) for sh in shapes_b]
    mask[0][30:60, 140:190] = 0
    soft = feather_model.feather_chain(states, labels, images, 0, mask)
    assert (soft != hard).any()
    only = feather_model.feather_pair(states[0], (images[labels[0]], images[labels[1]]), 0, mask[0])
    bx, by = int(states[0]["Bpts"][0][0]), int(states[0]["Bpts"][0][1])
    warped = cv2.warpPerspective(images[labels[1]], states[0]["cachedAH"], tuple(states[0]["ABSize"]))
    touched = feather_model.touched_mask(states[0]["cachedAH"], images[labels[1]].shape[:2], tuple(states[0]["ABSize"]))
    win = (slice(by + 30, by + 60), slice(bx + 140, bx + 190))
    assert np.array_equal(only[win][touched[win]], warped[win][touched[win]])


def _trimmed_super_chain(n, h, w, c, trim=(9, 5), kind="noise", frame_index=0):
    """A super-mode chain whose crops only trim ``trim`` pixels off every stage canvas, so that the pasted
    rectangles are CUT by the crops (their left / top edges fall outside the panorama) while seam bands
    survive.  The synthetic default limits (StitcherClass.py:344-351 on this camera layout) keep only the
    newest camera.  Returns (stitcher, oracle dict states, labels, images)."""
    from multicamera_stitching_b200 import Stitcher, synthetic
    images = synthetic.make_frames(n, h, w, c, frame_index, kind)
    st = Stitcher(images, super_mode=True)
    labels = list(st.img_labels)
    shapeB = tuple(images[labels[0]].shape)
    states = []
    for k in range(n - 1):
        H = synthetic.make_homography(k, h, w, shapeB[1])
        sb = st.stitchers[k]
        sb.set_homography(H, shapeA=images[labels[k + 1]].shape, shapeB=shapeB, xoffset=0, yoffset=0)
        sb.x_limits = [trim[0], sb.ABSize[0] - trim[0]]
        sb.y_limits = [trim[1], sb.ABSize[1] - trim[1]]
        shapeB = sb.result_shape()
        ost = stitcher_ref.new_state(sid=str(k), super_mode=True)
        for f in ("cachedBH", "cachedBINVH", "Bpts", "BimgSize", "cachedAH", "cachedAINVH", "Apts", "AimgSize",
                  "ABSize", "x_limits", "y_limits"):
            ost[f] = getattr(sb, f)
        states.append(ost)
    return st, states, labels, images


def test_feather_super_mode_crops_after_the_blended_paste():
    st, states, labels, images = _trimmed_super_chain(3, 120, 200, 3)
    soft = feather_model.feather_chain(states, labels, images, 2)
    hard = stitcher_ref.stitch_chain(states, labels, images)
    assert soft.shape == hard.shape and (soft != hard).any()
    # the crop of stage 0 cut the left / top edge of camera 0's pasted rectangle: no band there
    assert np.array_equal(soft[:, :20], hard[:, :20])


@pytest.mark.parametrize("seed", range(28))
def test_specification_reduces_to_the_overwrite_on_random_rigs(seed):
    """On the seeded random rigs (super-mode crops cutting the pasted rectangles): a one-pixel feather and maps
    of F everywhere are the reference's overwrite, and map values above F count as F."""
    from feather_cases import make_maps, rig, stage_shapes
    made = rig(seed)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    hard = stitcher_ref.stitch_chain(states, labels, images)
    assert np.array_equal(feather_model.feather_chain(states, labels, images, 0), hard)
    log2 = 1 + seed % 5
    shapes = stage_shapes(st, images, labels)
    full = make_maps(shapes, log2, "full")
    assert np.array_equal(feather_model.feather_chain(states, labels, images, log2, full), hard)
    over = make_maps(shapes, log2, "over", seed=seed)
    assert all(m.max() > (1 << log2) for m in over)
    clipped = [np.minimum(m, 1 << log2).astype(np.uint8) for m in over]
    soft = feather_model.feather_chain(states, labels, images, log2, over)
    assert np.array_equal(soft, feather_model.feather_chain(states, labels, images, log2, clipped))
    assert (soft != hard).any()


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w,c,log2", [
    (2, 64, 96, 3, 2), (3, 120, 200, 3, 3), (4, 90, 160, 1, 4), (4, 90, 160, 4, 1), (6, 270, 480, 3, 5),
])
def test_feather_kernel_matches_specification(cuda_device, n, h, w, c, log2):
    import torch
    st, states, labels, images = synthetic_chain(n, h, w, c, kind="noise", xoffset=2, yoffset=7)
    st.feather_log2 = log2
    ref = feather_model.feather_chain(states, labels, images, log2)
    got = st.stitch(images)
    assert got.shape == ref.shape
    assert np.array_equal(got, ref), int(np.abs(got.astype(int) - ref.astype(int)).max())
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    # one launch: the seam bands are BAND tiles of the tiled kernel (variant 4), blended in registers
    stats = plan.handle.tiled_stats()
    assert stats["band_fused"] == 1 and stats["band"] > 0, stats
    assert plan.handle.last_variant() == 4
    # batched, device-resident
    sets = [synthetic_chain(n, h, w, c, kind="noise", frame_index=f)[3] for f in range(3)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    out = st.stitch_batch(batch).cpu().numpy()
    for f in range(3):
        assert np.array_equal(out[f], feather_model.feather_chain(states, labels, sets[f], log2))
    # width one = the reference's overwrite through the regular kernels
    st.feather_log2 = 0
    assert np.array_equal(st.stitch(images), stitcher_ref.stitch_chain(states, labels, images))


@pytest.mark.gpu
def test_feather_fused_launch_count_and_window_uploads(cuda_device):
    """The fused form is ONE kernel launch per call, and it keeps the visible-window uploads: the source windows
    the plan reports cover what the band samples read (a frame poisoned outside them gives the same panorama)."""
    import torch
    from multicamera_stitching_b200 import _cabi
    n, h, w, c, log2 = 4, 180, 320, 3, 3
    st, states, labels, images = synthetic_chain(n, h, w, c, kind="noise")
    st.feather_log2 = log2
    ref = feather_model.feather_chain(states, labels, images, log2)
    assert np.array_equal(st.stitch(images), ref)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    batch = {l: torch.from_numpy(images[l][None]).to(cuda_device) for l in labels}
    before = _cabi.launch_count()
    st.stitch_batch(batch)
    assert _cabi.launch_count() - before == 1
    bands = plan.upload_bands()
    poisoned = {}
    some_hidden = False
    for k, l in enumerate(labels):
        row, rows, copies = bands[k]
        keep = np.zeros((rows, row), bool)
        for cp in copies:
            keep[cp["y0"]:cp["y0"] + cp["rows"], cp["b0"]:cp["b0"] + cp["nbytes"]] = True
        some_hidden |= not keep.all()
        flat = images[l].reshape(rows, row).copy()
        flat[~keep] = 255 - flat[~keep]
        poisoned[l] = torch.from_numpy(flat.reshape(images[l].shape)[None]).to(cuda_device)
    assert some_hidden
    assert np.array_equal(st.stitch_batch(poisoned)[0].cpu().numpy(), ref)


@pytest.mark.gpu
def test_feather_two_pass_form_still_matches(cuda_device, monkeypatch):
    """$MCS_TILED_BAND=0 (and plans the fused form cannot express: more than two outer layers per tile, feathers over
    more than 32 pixels) composite with the overwrite kernel and re-evaluate the bands in a second pass."""
    n, h, w, c = 3, 120, 200, 3
    st, states, labels, images = synthetic_chain(n, h, w, c, kind="noise", xoffset=2, yoffset=7)
    monkeypatch.setenv("MCS_TILED_BAND", "0")
    st.feather_log2 = 3
    assert np.array_equal(st.stitch(images), feather_model.feather_chain(states, labels, images, 3))
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.tiled_stats()["band_fused"] == 0 and plan.handle.last_variant() == 3
    monkeypatch.delenv("MCS_TILED_BAND")
    st.__dict__.pop("_engine", None)
    st.feather_log2 = 6   # 64 pixels: beyond the six weight bits of the overlay descriptors
    assert np.array_equal(st.stitch(images), feather_model.feather_chain(states, labels, images, 6))
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.tiled_stats()["band_fused"] == 0 and plan.handle.last_variant() == 3


@pytest.mark.gpu
def test_feather_on_the_fly_band_kernel_and_many_frames(cuda_device, monkeypatch):
    """The plan-time sample table (default) and the on-the-fly band kernel (tables over 2 GB,
    or $MCS_FEATHER_TABLE=0) give the same panoramas; 11 frames = one full and one partial
    group of the table kernel's 8 frames per thread."""
    import torch
    n, h, w, c, log2 = 4, 90, 160, 3, 3
    st, states, labels, images = synthetic_chain(n, h, w, c, kind="noise", xoffset=2, yoffset=7)
    sets = [synthetic_chain(n, h, w, c, kind="noise", frame_index=f)[3] for f in range(11)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    refs = [feather_model.feather_chain(states, labels, s, log2) for s in sets]
    monkeypatch.setenv("MCS_TILED_BAND", "0")      # the two-pass form is what this test is about
    for table in ("1", "0"):
        monkeypatch.setenv("MCS_FEATHER_TABLE", table)
        st.__dict__.pop("_engine", None)          # new plan: the switch is read when the plan is built
        st.feather_log2 = log2
        out = st.stitch_batch(batch).cpu().numpy()
        for f in range(11):
            assert np.array_equal(out[f], refs[f]), (table, f)


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w,c,log2,super_mode", [
    (3, 120, 200, 3, 3, False), (4, 90, 160, 1, 5, False), (3, 120, 200, 4, 0, False), (5, 135, 240, 3, 2, False),
    (3, 120, 200, 3, 2, True), (4, 180, 320, 3, 3, True),
])
def test_weight_maps_match_the_specification(cuda_device, n, h, w, c, log2, super_mode):
    """Per-stage u8 weight maps (mcs_plan_set_blend), blended in registers by the BAND tiles; with
    feather_log2 == 0 they are {0, 1} masks; in super mode distances / maps refer to the pasted rectangles."""
    import torch
    if super_mode:
        st, states, labels, images = _trimmed_super_chain(n, h, w, c)
    else:
        st, states, labels, images = synthetic_chain(n, h, w, c, kind="noise")
    maps = _random_weights(states, images, labels, log2, seed=n)
    st.feather_log2 = log2
    st.blend_weights = maps
    ref = feather_model.feather_chain(states, labels, images, log2, maps)
    got = st.stitch(images)
    assert got.shape == ref.shape
    assert np.array_equal(got, ref), int(np.abs(got.astype(int) - ref.astype(int)).max())
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.tiled_stats()["band_fused"] == 1 and plan.handle.last_variant() == 4
    from multicamera_stitching_b200 import synthetic
    sets = [synthetic.make_frames(n, h, w, c, f, "noise") for f in range(3)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    out = st.stitch_batch(batch).cpu().numpy()
    for f in range(3):
        assert np.array_equal(out[f], feather_model.feather_chain(states, labels, sets[f], log2, maps))
    # some maps missing: those stages fall back to the ramp
    if log2 > 0:
        st.blend_weights = [maps[0]] + [None] * (n - 2)
        assert np.array_equal(st.stitch(images), feather_model.feather_chain(states, labels, images, log2,
                                                                              [maps[0]] + [None] * (n - 2)))


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w,c,log2", [(3, 120, 200, 3, 3), (4, 180, 320, 3, 2), (5, 135, 240, 1, 4)])
def test_feather_ramp_in_super_mode(cuda_device, n, h, w, c, log2):
    st, states, labels, images = _trimmed_super_chain(n, h, w, c)
    st.feather_log2 = log2
    ref = feather_model.feather_chain(states, labels, images, log2)
    hard = stitcher_ref.stitch_chain(states, labels, images)
    assert (ref != hard).any()
    got = st.stitch(images)
    assert got.shape == ref.shape and np.array_equal(got, ref)
    # and the default synthetic super-mode limits (only the newest camera survives each crop)
    st2, states2, labels2, images2 = synthetic_chain(n, h, w, c, kind="noise", super_mode=True)
    st2.feather_log2 = log2
    assert np.array_equal(st2.stitch(images2), feather_model.feather_chain(states2, labels2, images2, log2))


@pytest.mark.gpu
def test_fused_bands_over_several_frame_blocks(cuda_device, monkeypatch):
    """BAND chunks of frame block b + 1 follow the COPY / ZERO chunks of block b in the sweep: the box issuer
    enters a BAND chunk only when the consumers get there.  11 frames in blocks of 4."""
    import torch
    monkeypatch.setenv("MCS_TILED_FRAME_BLOCK", "4")
    n, h, w, c, log2 = 5, 270, 480, 3, 3
    st, states, labels, images = synthetic_chain(n, h, w, c, kind="noise", xoffset=2, yoffset=7)
    st.feather_log2 = log2
    sets = [synthetic_chain(n, h, w, c, kind="noise", frame_index=f)[3] for f in range(11)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    out = st.stitch_batch(batch).cpu().numpy()
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.last_variant() == 4
    for f in range(11):
        assert np.array_equal(out[f], feather_model.feather_chain(states, labels, sets[f], log2)), f


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [0.62, 0.45])
def test_fused_bands_with_large_source_boxes(cuda_device, scale):
    """Minifying cameras: the staged source boxes grow (24 KB, 39 KB) until only three fit the ring - at the smaller
    scale with one CTA per SM - so a BAND unit's two boxes per frame leave the issuer a look-ahead of one box.
    Against the specification, single frames and a batch."""
    import torch
    from multicamera_stitching_b200 import Stitcher, synthetic
    n, h, w, c, log2 = 3, 360, 640, 3, 3
    images = synthetic.make_frames(n, h, w, c, 0, "noise")
    st = Stitcher(images)
    labels = list(st.img_labels)
    states = []
    shapeB = images[labels[0]].shape
    for k in range(n - 1):
        H = np.array([[scale, 0.02, shapeB[1] - 0.4 * w * scale], [-0.012, scale, 9.0 * (1 if k % 2 == 0 else -1)],
                      [1e-5, -0.5e-5, 1.0]])
        st.stitchers[k].set_homography(H, shapeA=images[labels[k + 1]].shape, shapeB=shapeB, xoffset=0, yoffset=0)
        ost = stitcher_ref.new_state(sid=str(k))
        stitcher_ref.geometry_from_homography(ost, H, images[labels[k + 1]].shape, shapeB, 0, 0)
        states.append(ost)
        shapeB = st.stitchers[k].result_shape()
    st.feather_log2 = log2
    ref = feather_model.feather_chain(states, labels, images, log2)
    got = st.stitch(images)
    assert np.array_equal(got, ref)
    sets = [synthetic.make_frames(n, h, w, c, f, "noise") for f in range(5)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    out = st.stitch_batch(batch).cpu().numpy()
    for f in range(5):
        assert np.array_equal(out[f], feather_model.feather_chain(states, labels, sets[f], log2)), f
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    stats = plan.handle.tiled_stats()
    assert plan.handle.last_variant() in (3, 4) and (stats["band_fused"] == 1) == (plan.handle.last_variant() == 4)
