"""GPU parity tests of the fused warp+paste kernel, through the C ABI.

Checker: the reference's own sequential chain driven through cv2
(oracle/stitcher_ref.py = StitcherClass.py:114-136, :211-256) and the
transparent integer model (oracle/composite_model.py).  Bar: uint8 within
+-1 LSB, >= 99.9 % of values bit-exact (BASELINE.json); the kernel is expected
to be 100 % exact and the tests say so where they can.
"""
import numpy as np
import pytest
import torch

from helpers import compare_u8, synthetic_chain
from oracle import composite_model, stitcher_ref

pytestmark = pytest.mark.gpu

MAX_ABS = 1          # +-1 LSB
MIN_EXACT = 0.999    # >= 99.9 % bit-exact


def _check(got, ref, exact=True):
    mx, frac = compare_u8(got, ref)
    assert mx <= MAX_ABS and frac >= MIN_EXACT, (mx, frac)
    if exact:
        assert mx == 0, (mx, frac)


@pytest.mark.parametrize("n,h,w,c,kind", [
    (3, 720, 1280, 3, "smooth"),     # BASELINE config 1
    (3, 720, 1280, 3, "noise"),      # stress: one bucket flip = several grey levels
    (4, 240, 320, 1, "noise"),       # 2-D grayscale frames (MediaPlayer feeds those)
    (2, 97, 131, 3, "noise"),        # odd sizes, unaligned pitches
    (5, 120, 50, 3, "noise"),        # frames narrower than one 64-column block
])
def test_chain_matches_cv2(cuda_device, n, h, w, c, kind):
    st, states, labels, images = synthetic_chain(n, h, w, c, kind=kind, use_points_first=True)
    ref = stitcher_ref.stitch_chain(states, labels, images)
    got = st.stitch(images)
    assert isinstance(got, np.ndarray) and got.dtype == np.uint8
    _check(got, ref)


@pytest.mark.parametrize("xoffset,yoffset", [(0, 0), (10, 10), (3, 25)])
def test_offsets_and_super_mode(cuda_device, xoffset, yoffset):
    for super_mode in (False, True):
        st, states, labels, images = synthetic_chain(3, 180, 320, 3, super_mode=super_mode, kind="noise",
                                                     xoffset=xoffset, yoffset=yoffset)
        ref = stitcher_ref.stitch_chain(states, labels, images)
        got = st.stitch(images)
        _check(got, ref)


def test_pair_stitch_matches_cv2(cuda_device):
    st, states, labels, images = synthetic_chain(2, 200, 300, 3, kind="noise")
    pair = (images[labels[0]], images[labels[1]])
    ref = stitcher_ref.stitch_pair(states[0], pair)
    got = st.stitchers[0].stitch(pair)
    _check(got, ref)


def test_cuda_tensor_in_cuda_tensor_out_and_batch(cuda_device):
    st, states, labels, images = synthetic_chain(3, 144, 256, 3, kind="noise")
    dev = {l: torch.from_numpy(images[l]).to(cuda_device) for l in labels}
    out = st.stitch(dev)
    assert isinstance(out, torch.Tensor) and out.is_cuda
    ref0 = stitcher_ref.stitch_chain(states, labels, images)
    _check(out.cpu().numpy(), ref0)
    # batch of 3 different frame-sets in one launch
    sets = []
    for f in range(3):
        _, _, _, im = synthetic_chain(3, 144, 256, 3, kind="noise", frame_index=f)
        sets.append(im)
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    outb = st.stitch_batch(batch)
    assert outb.shape[0] == 3
    for f in range(3):
        _check(outb[f].cpu().numpy(), stitcher_ref.stitch_chain(states, labels, sets[f]))


def test_four_channel_against_model(cuda_device):
    # cv2 also handles 4 channels; compare with both checkers
    st, states, labels, images = synthetic_chain(3, 100, 160, 4, kind="noise")
    ref = stitcher_ref.stitch_chain(states, labels, images)
    got = st.stitch(images)
    _check(got, ref)


def test_strided_sources_and_padded_output(cuda_device):
    st, states, labels, images = synthetic_chain(3, 96, 200, 3, kind="noise")
    ref = stitcher_ref.stitch_chain(states, labels, images)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    srcs = []
    for l in labels:
        h, w, c = images[l].shape
        big = torch.zeros((h, w + 13, c), dtype=torch.uint8, device=cuda_device)
        big[:, 5:5 + w] = torch.from_numpy(images[l]).to(cuda_device)
        srcs.append(big[:, 5:5 + w])           # row pitch != w*c, base not 16-byte aligned
    out = plan.new_output(pitch_align=256)
    guard = out.storage_offset()
    assert guard == 0
    res = plan.run(srcs, out=out)
    _check(res.cpu().numpy(), ref)


def test_owned_pixels_and_algorithmic_bytes(cuda_device):
    st, states, labels, images = synthetic_chain(3, 180, 320, 3, kind="smooth")
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    _, owned_model = composite_model.composite(plan.flat.layers, plan.out_w, plan.out_h,
                                               [images[l] for l in labels])
    assert plan.owned_pixels() == owned_model
    assert plan.algorithmic_bytes() == plan.out_w * plan.out_h * 3 + 3 * sum(owned_model)


def test_singular_and_identity_homographies(cuda_device):
    rng = np.random.default_rng(5)
    a = rng.integers(0, 256, (80, 120, 3), dtype=np.uint8)
    b = rng.integers(0, 256, (80, 120, 3), dtype=np.uint8)
    from multicamera_stitching_b200 import Stitcher
    for H in (np.eye(3), np.array([[1, 0, 37.0], [0, 1, -12.0], [0, 0, 1]]),
              np.array([[0.5, 0.3, 10.0], [-0.4, 0.6, 50.0], [1e-3, -5e-4, 1]])):
        st = Stitcher({"A": b, "B": a})
        st.stitchers[0].set_homography(H, a.shape, b.shape, 0, 0)
        ost = stitcher_ref.new_state()
        stitcher_ref.geometry_from_homography(ost, H, a.shape, b.shape, 0, 0)
        ref = stitcher_ref.stitch_pair(ost, (b, a))
        got = st.stitchers[0].stitch((b, a))
        _check(got, ref)


def test_singular_homography_through_the_plan(cuda_device):
    """cv2.invert zero-fills a singular matrix, so every pixel samples src(0,0)."""
    import cv2
    from multicamera_stitching_b200.engine import CompiledPlan
    from multicamera_stitching_b200.plan import FlatPlan, Layer, LAYER_WARP
    rng = np.random.default_rng(6)
    a = rng.integers(0, 256, (40, 60, 3), dtype=np.uint8)
    M = np.array([[1, 2, 3.0], [2, 4, 6.0], [0, 0, 1]])
    flat = FlatPlan([Layer(0, LAYER_WARP, M, 0, 0, (0, 0, 50, 30), (40, 60))], 50, 30, 3, 3)
    plan = CompiledPlan(flat, cuda_device)
    got = plan.run([torch.from_numpy(a).to(cuda_device)]).cpu().numpy()
    assert np.array_equal(got, cv2.warpPerspective(a, M, (50, 30)))


def _run_variant(st, labels, images, device, variant):
    """Composite through a pinned kernel variant (1 = gather, 2 = tiled/TMA)."""
    plan = st.plan([images[l].shape for l in labels], device)
    if variant == 2:
        assert plan.handle.tiled_status() == "", plan.handle.tiled_status()
    plan.handle.force_variant(variant)
    try:
        dev = {l: torch.from_numpy(images[l]).to(device) for l in labels}
        out = st.stitch(dev).cpu().numpy()
        assert plan.handle.last_variant() == variant
    finally:
        plan.handle.force_variant(0)
    return out


@pytest.mark.parametrize("n,h,w,c,super_mode,off", [
    (3, 720, 1280, 3, False, 0),
    (3, 360, 640, 3, True, 0),
    (4, 240, 320, 1, False, 7),
    (4, 240, 320, 4, False, 3),
    (6, 270, 480, 3, False, 0),
    (8, 135, 240, 3, False, 5),
    (2, 64, 48, 3, False, 0),
])
def test_tiled_variant_matches_cv2_and_gather(cuda_device, n, h, w, c, super_mode, off):
    st, states, labels, images = synthetic_chain(n, h, w, c, super_mode=super_mode, kind="noise",
                                                 xoffset=off, yoffset=off, use_points_first=True)
    ref = stitcher_ref.stitch_chain(states, labels, images)
    tiled = _run_variant(st, labels, images, cuda_device, 2)
    gather = _run_variant(st, labels, images, cuda_device, 1)
    _check(gather, ref)
    _check(tiled, ref)


@pytest.mark.parametrize("name,H", [
    ("rot30", [[0.866, -0.5, 150.0], [0.5, 0.866, -20.0], [0, 0, 1]]),
    ("rot90", [[0.0, -1.0, 400.0], [1.0, 0.0, 10.0], [0, 0, 1]]),
    ("down", [[0.45, 0.02, 180.0], [0.01, 0.5, 30.0], [1e-5, 0, 1]]),
    ("up", [[2.2, 0.1, 100.0], [-0.1, 2.4, 50.0], [1e-4, 2e-4, 1]]),
    ("persp", [[1.0, 0.05, 120.0], [0.02, 1.1, 5.0], [6e-4, -2e-4, 1]]),
    ("far_away", [[1.0, 0.0, 5000.0], [0.0, 1.0, 3000.0], [0, 0, 1]]),
    ("flip", [[-1.0, 0.0, 500.0], [0.0, 1.0, 0.0], [0, 0, 1]]),
])
def test_tiled_variant_general_homographies(cuda_device, name, H):
    from multicamera_stitching_b200 import Stitcher
    rng = np.random.default_rng(11)
    b = rng.integers(0, 256, (160, 256, 3), dtype=np.uint8)
    a = rng.integers(0, 256, (192, 320, 3), dtype=np.uint8)
    st = Stitcher({"A": b, "B": a})
    st.stitchers[0].set_homography(np.array(H), a.shape, b.shape, 0, 0)
    ost = stitcher_ref.new_state()
    stitcher_ref.geometry_from_homography(ost, np.array(H), a.shape, b.shape, 0, 0)
    ref = stitcher_ref.stitch_pair(ost, (b, a))
    images = {"A": b, "B": a}
    labels = ["A", "B"]
    plan = st.plan([b.shape, a.shape], cuda_device)
    if plan.handle.tiled_status() == "":
        _check(_run_variant(st, labels, images, cuda_device, 2), ref)
    _check(_run_variant(st, labels, images, cuda_device, 1), ref)
    _check(st.stitch(images), ref)


def test_tiled_variant_unaligned_destination(cuda_device):
    st, states, labels, images = synthetic_chain(3, 144, 256, 3, kind="noise")
    ref = stitcher_ref.stitch_chain(states, labels, images)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    srcs = [torch.from_numpy(images[l]).to(cuda_device) for l in labels]
    plan.handle.force_variant(2)
    try:
        for pad, shift in ((1, 0), (7, 3), (16, 5), (64, 1)):
            row = plan.out_w * 3 + pad
            buf = torch.full((plan.out_h * row + 64,), 0xAB, dtype=torch.uint8, device=cuda_device)
            out = torch.as_strided(buf, (plan.out_h, plan.out_w, 3), (row, 3, 1), storage_offset=shift)
            plan.run(srcs, out=out)
            _check(out.cpu().numpy(), ref)
            # padding bytes between rows stay untouched
            flat = buf.cpu().numpy()
            assert (flat[:shift] == 0xAB).all()
            gap = flat[shift:shift + plan.out_h * row].reshape(plan.out_h, row)[:, plan.out_w * 3:]
            assert (gap == 0xAB).all()
    finally:
        plan.handle.force_variant(0)


def test_tiled_variant_batch(cuda_device):
    st, states, labels, images = synthetic_chain(3, 144, 256, 3, kind="noise")
    sets = []
    for f in range(5):
        _, _, _, im = synthetic_chain(3, 144, 256, 3, kind="noise", frame_index=f)
        sets.append(im)
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    plan.handle.force_variant(2)
    try:
        outb = st.stitch_batch(batch)
    finally:
        plan.handle.force_variant(0)
    for f in range(5):
        _check(outb[f].cpu().numpy(), stitcher_ref.stitch_chain(states, labels, sets[f]))


def test_full_size_config2_vs_cv2(cuda_device):
    """BASELINE config 2 at full size (6 x 1080p): cv2 needs ~0.1 s."""
    st, states, labels, images = synthetic_chain(6, 1080, 1920, 3, kind="smooth")
    ref = stitcher_ref.stitch_chain(states, labels, images)
    got = st.stitch(images)
    _check(got, ref)
    st, states, labels, images = synthetic_chain(6, 1080, 1920, 3, kind="noise")
    _check(st.stitch(images), stitcher_ref.stitch_chain(states, labels, images))


def test_full_size_config3_vs_cv2(cuda_device):
    """BASELINE config 3 at full size (8 x 2160p into a wide canvas)."""
    st, states, labels, images = synthetic_chain(8, 2160, 3840, 3, kind="smooth")
    ref = stitcher_ref.stitch_chain(states, labels, images)
    got = st.stitch(images)
    _check(got, ref)
    # size-independent property: compositing is idempotent on its own inputs and
    # camera 0 is pasted verbatim
    l0 = st.plan([images[l].shape for l in labels], cuda_device).flat.layers[0]
    x0, y0, x1, y1 = l0.rect
    assert np.array_equal(got[y0:y1, x0:x1], images[labels[0]][y0 - l0.oy:y1 - l0.oy, x0 - l0.ox:x1 - l0.ox])


@pytest.mark.parametrize("frame_block,n_frames,pitch_align", [
    (1, 5, 1), (4, 11, 128), (4, 8, 1), (32, 11, 128), (3, 7, 32),
])
def test_tiled_variant_frame_blocks(cuda_device, monkeypatch, frame_block, n_frames, pitch_align):
    """The work split of the tiled kernel: frame blocks (last one shorter), round-robin cells plus
    leftover runs, padded and dense panorama pitch - every frame of the batch must equal the cv2
    chain on that frame's inputs."""
    monkeypatch.setenv("MCS_TILED_FRAME_BLOCK", str(frame_block))
    st, states, labels, images = synthetic_chain(6, 270, 480, 3, kind="noise", xoffset=4, yoffset=9)
    sets = [synthetic_chain(6, 270, 480, 3, kind="noise", frame_index=f)[3] for f in range(n_frames)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.tiled_status() == "", plan.handle.tiled_status()
    out = plan.new_output(n_frames, pitch_align=pitch_align)
    out.fill_(0xCD)
    plan.handle.force_variant(2)
    try:
        st.stitch_batch(batch, out=out)
        assert plan.handle.last_variant() == 2
    finally:
        plan.handle.force_variant(0)
    got = out.cpu().numpy()
    for f in range(n_frames):
        _check(got[f], stitcher_ref.stitch_chain(states, labels, sets[f]))


def test_batch_equals_single_frames_config2(cuda_device):
    """Size-independent property at BASELINE config 2's full size: a batched launch (several
    frames per chunk, leftover runs split between CTAs) gives, frame by frame, exactly what
    one-frame launches give."""
    st, states, labels, images = synthetic_chain(6, 1080, 1920, 3, kind="smooth")
    sets = [synthetic_chain(6, 1080, 1920, 3, kind="smooth", frame_index=f)[3] for f in range(3)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    out = st.stitch_batch(batch, out=plan.new_output(3, pitch_align=128))
    assert plan.handle.last_variant() == 2
    for f in range(3):
        single = st.stitch({l: batch[l][f] for l in labels})
        assert torch.equal(out[f], single)
    _check(out[0].cpu().numpy(), stitcher_ref.stitch_chain(states, labels, sets[0]))


def test_rows_that_are_not_16_byte_multiples_still_take_the_tiled_kernel(cuda_device):
    """360-pixel BGR rows are 1080 bytes: TMA cannot address them, the gather kernel is ~5x slower,
    so the engine realigns such frames into a pitched scratch buffer (one device-side copy) and
    launches the tiled kernel."""
    st, states, labels, images = synthetic_chain(4, 200, 360, 3, kind="noise")
    ref = stitcher_ref.stitch_chain(states, labels, images)
    _check(st.stitch(images), ref)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.tiled_status() == "" and plan.handle.last_variant() == 2
    sets = [synthetic_chain(4, 200, 360, 3, kind="noise", frame_index=f)[3] for f in range(3)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    outb = st.stitch_batch(batch)
    assert plan.handle.last_variant() == 2
    for f in range(3):
        _check(outb[f].cpu().numpy(), stitcher_ref.stitch_chain(states, labels, sets[f]))


@pytest.mark.parametrize("n,h,w,c", [(3, 120, 131, 3), (2, 97, 403, 1), (4, 90, 854, 3)])
def test_rows_that_are_not_4_byte_multiples_take_the_tiled_kernel_through_zero_padded_rows(cuda_device, n, h, w, c):
    """A 131-pixel BGR row is 393 bytes.  The engine's scratch rows are zero-padded, it promises
    that to the plan (mcs_plan_promise_padded_rows), and the pad bytes stand in for the
    BORDER_CONSTANT taps right of the image."""
    st, states, labels, images = synthetic_chain(n, h, w, c, kind="noise")
    ref = stitcher_ref.stitch_chain(states, labels, images)
    _check(st.stitch(images), ref)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.rows_need_padding() and plan.handle.last_variant() == 2
    dev = {l: torch.from_numpy(images[l]).to(cuda_device) for l in labels}
    _check(st.stitch(dev).cpu().numpy(), ref)
    # without the promise the same plan falls back to the gather kernel (direct C-ABI callers)
    plan.handle.promise_padded_rows(False)
    _check(st.stitch(dev).cpu().numpy(), ref)
    assert plan.handle.last_variant() == 1
    plan.handle.promise_padded_rows(True)


def test_realigned_sources_with_odd_frame_strides(cuda_device):
    """Batched views whose frames are not a whole number of rows apart still go through the scratch
    copy (frame by frame) and the tiled kernel."""
    st, states, labels, images = synthetic_chain(3, 96, 131, 3, kind="noise")
    sets = [synthetic_chain(3, 96, 131, 3, kind="noise", frame_index=f)[3] for f in range(3)]
    batch = {}
    for l in labels:
        h, w, c = images[l].shape
        flat = torch.zeros(3 * (h * w * c + 7) + 5, dtype=torch.uint8, device=cuda_device)
        view = torch.as_strided(flat, (3, h, w, c), (h * w * c + 7, w * c, c, 1), 5)
        view.copy_(torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device))
        batch[l] = view
    out = st.stitch_batch(batch)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.last_variant() == 2
    for f in range(3):
        _check(out[f].cpu().numpy(), stitcher_ref.stitch_chain(states, labels, sets[f]))


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w", [(8, 1080, 1920), (8, 2160, 3840)])
def test_full_size_ownership_partition(cuda_device, n, h, w):
    """Size-independent property at BASELINE.json's full sizes (the default bench geometry and config 3), no oracle
    involved: with camera k painted in the constant colour (c_k, 255 - c_k, 128), bilinear resampling of a constant
    is that constant wherever all four taps lie inside the source, and a border pixel (taps mixed with the zero
    fill) scales all three channels by the same weight, so it matches no camera's colour.  The panorama is then
    made of background zeros, camera colours and a thin ring of border mixes, and the count of every colour is
    what ``mcs_plan_owned_pixels`` - the figure behind the roofline's algorithmic bytes - reports, up to that ring."""
    import torch
    st, states, labels, images = synthetic_chain(n, h, w, 3)
    colours = [(16 + 24 * k, 255 - (16 + 24 * k), 128) for k in range(n)]
    frames = {}
    for k, l in enumerate(labels):
        f = torch.empty((1, h, w, 3), dtype=torch.uint8, device=cuda_device)
        for c in range(3):
            f[..., c] = colours[k][c]
        frames[l] = f
    pano = st.stitch_batch(frames)[0].to(torch.int32)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.last_variant() == 2
    owned = plan.owned_pixels()
    layer_of_cam = {l.cam: i for i, l in enumerate(plan.flat.layers)}
    key = pano[..., 0] * 65536 + pano[..., 1] * 256 + pano[..., 2]
    accounted = int((key == 0).sum())
    ring_total = 0
    for k in range(n):
        ck = colours[k][0] * 65536 + colours[k][1] * 256 + colours[k][2]
        exact = int((key == ck).sum())
        own = owned[layer_of_cam[k]]
        ring = 2 * (h + w) * 3          # owned pixels whose taps straddle the source border
        assert own - ring <= exact <= own, (k, exact, own)
        ring_total += own - exact
        accounted += exact
    # what is neither background nor a camera colour is a border mix of an owned pixel
    assert int(key.numel()) - accounted <= ring_total
    assert int((key == 0).sum()) >= int(key.numel()) - sum(owned)


@pytest.mark.gpu
def test_full_size_blend_reduces_to_the_overwrite(cuda_device):
    """Size-independent property of the blend modes at config 2's full size: weight maps that are F everywhere
    are the reference's overwrite (StitcherClass.py:240-241), bit for bit, through the BAND-aware kernel."""
    import torch
    st, states, labels, images = synthetic_chain(6, 1080, 1920, 3)
    frames = {l: torch.from_numpy(images[l][None]).to(cuda_device) for l in labels}
    hard = st.stitch_batch(frames).clone()
    shapes = []
    shapeB = images[labels[0]].shape
    for sb in st.stitchers:
        shapes.append(tuple(shapeB[:2]))
        shapeB = sb.result_shape()
    st.feather_log2 = 4
    st.blend_weights = [np.full(sh, 16, np.uint8) for sh in shapes]
    assert torch.equal(st.stitch_batch(frames), hard)
    # a real ramp on one stage only changes pixels within F - 1 of that stage's pasted rectangle border
    st.blend_weights = None
    soft = st.stitch_batch(frames)
    changed = (soft != hard).any(dim=-1)[0]
    assert bool(changed.any())
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.last_variant() == 4
    # the seam band of stage k lies within F - 1 = 15 pixels inside the border of layer k - 1's rectangle
    inner_ok = torch.zeros_like(changed)
    for l in plan.flat.layers[:-1]:
        x0, y0, x1, y1 = l.rect
        band = torch.zeros_like(changed)
        band[y0:y1, x0:x1] = True
        if y1 - y0 > 30 and x1 - x0 > 30:
            band[y0 + 15:y1 - 15, x0 + 15:x1 - 15] = False
        inner_ok |= band
    assert not bool((changed & ~inner_ok).any())


@pytest.mark.gpu
@pytest.mark.parametrize("n_frames", [65, 67, 130])
def test_frame_counts_whose_last_block_is_shorter_than_the_split(cuda_device, n_frames):
    """64-frame blocks with 1-3 frames left over: the launcher must not cut the last tiles of such a block into
    chunks without frames (tests/test_issuer_protocol.py: the box issuer would starve).  Every frame against the
    single-frame result."""
    import torch
    st, states, labels, images = synthetic_chain(4, 120, 200, 3, kind="noise")
    ref = stitcher_ref.stitch_chain(states, labels, images)
    batch = {l: torch.from_numpy(images[l]).to(cuda_device)[None].expand(n_frames, -1, -1, -1).contiguous() for l in labels}
    out = st.stitch_batch(batch)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.last_variant() == 2
    want = torch.from_numpy(ref).to(cuda_device)
    assert bool((out == want[None]).all())


@pytest.mark.parametrize("n,h,w,c,super_mode", [(3, 97, 131, 3, False), (3, 96, 132, 3, False), (4, 120, 200, 1, False),
                                                  (3, 90, 160, 4, True)])
def test_gather_variant_batches(cuda_device, monkeypatch, n, h, w, c, super_mode):
    """The fallback kernel loops the frames of a launch inside its threads (16 per thread, the rest through
    grid.z): batches around that block size, frame by frame against the cv2 chain - with rows that are and are
    not multiples of four bytes (aligned word loads or byte loads for the taps), and with the byte loads forced
    ($MCS_GATHER_BYTES)."""
    st, states, labels, images = synthetic_chain(n, h, w, c, kind="noise", super_mode=super_mode)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    try:
        plan.handle.force_variant(1)
        for F in (1, 15, 16, 17, 35):
            sets = [synthetic_chain(n, h, w, c, kind="noise", super_mode=super_mode, frame_index=f % 5)[3] for f in range(F)]
            batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
            refs = [stitcher_ref.stitch_chain(states, labels, sets[f]) for f in range(min(F, 5))]
            for mode in ("", "MCS_GATHER_BYTES"):
                monkeypatch.delenv("MCS_GATHER_BYTES", raising=False)
                if mode:
                    monkeypatch.setenv(mode, "1")
                # dense panorama rows, and rows padded to a multiple of four bytes
                for out in (None, plan.new_output(F, pitch_align=4)):
                    got = st.stitch_batch(batch, out=out).cpu().numpy()
                    assert plan.handle.last_variant() == 1
                    for f in range(F):
                        assert np.array_equal(got[f], refs[f % 5]), (F, f, mode, out is None)
    finally:
        plan.handle.force_variant(0)
