"""Camera-weighted blend on the GPU, fuzzed: mcs_stitch_weighted_kernel and the plan-time contributor
counter against the layer model of oracle/camera_weight_model.py, bit for bit.

- the seeded random rigs of the overwrite fuzz (tests/random_rigs.py), super-mode crops trimmed so that
  several cameras blend, under every map kind;
- those rigs through strided sources and a poisoned output, at frame counts on both sides of the
  kernel's 16-frame loop and of grid.z steps, on the word path and the byte path;
- the 4-contributor limit from both sides, down to one isolated pixel with 5 contributors at the edges
  of the counter's 32 x 16 blocks and of the panorama;
- the smallest and largest divisors, exact-half roundings of weights and values;
- REMAP layers (undistortion and random fixed-point maps with taps outside the source);
- the map pitch of the C ABI."""
import ctypes

import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, layer_model, make_maps
from multicamera_stitching_b200 import _cabi, prewarp
from multicamera_stitching_b200.plan import LAYER_COPY, LAYER_REMAP, LAYER_WARP, FlatPlan, Layer
from oracle import camera_weight_model, composite_model
from random_rigs import mirrored, random_chain

pytestmark = pytest.mark.gpu

MAX = camera_weight_model.MAX_CONTRIBUTORS
SEEDS = range(28)

# what the file exercised, asserted by the last test
COVERED = {"rigs_3plus": set(), "mirrored": set(), "channels": set(), "paths": set(), "frames": set(),
           "accepted_most4": 0, "refused_isolated5": 0}


def _rig(seed):
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    return made


def _channels(images, labels):
    a = images[labels[0]]
    return 1 if a.ndim == 2 else a.shape[2]


def _dev(torch, arrays, device):
    return [torch.from_numpy(np.ascontiguousarray(a)).to(device) for a in arrays]


def _blend(flat, frames, maps):
    return camera_weight_model.blend(flat.layers, flat.out_w, flat.out_h, frames, maps)


def _check_accepted(plan, flat, frames, maps, device):
    """Run ``plan`` (camera weights set) on ``frames``; it must equal the layer model.  Returns the model's most."""
    import torch
    ref, contrib, most = _blend(flat, frames, maps)
    got = plan.run(_dev(torch, frames, device)).cpu().numpy()
    assert plan.handle.last_variant() == 5
    assert np.array_equal(got, ref), int(np.abs(got.astype(int) - ref.astype(int)).max())
    assert plan.owned_pixels() == contrib
    return most


# ---- a. random rigs ------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", SEEDS)
def test_random_rig_matches_the_layer_model(cuda_device, seed):
    import torch
    st, states, labels, images = _rig(seed)
    kind = MAP_KINDS[seed % len(MAP_KINDS)]
    maps = make_maps(images, labels, kind, seed=seed)
    ref, contrib, most = layer_model(st, labels, images, maps)
    st.camera_weights = maps
    if most > MAX:
        with pytest.raises(_cabi.McsError, match="code -3"):
            st.stitch(images)
        return
    got = st.stitch(images)
    assert got.shape == ref.shape and np.array_equal(got, ref), int(np.abs(got.astype(int) - ref.astype(int)).max())
    dev = {l: torch.from_numpy(images[l]).to(cuda_device) for l in labels}
    assert np.array_equal(st.stitch(dev).cpu().numpy(), ref)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.last_variant() == 5
    assert plan.owned_pixels() == contrib
    assert plan.algorithmic_bytes() == plan.out_w * plan.out_h * plan.channels + plan.channels * sum(contrib)
    if most >= 3:
        COVERED["rigs_3plus"].add(seed)
    if mirrored(seed):
        COVERED["mirrored"].add(seed)
    COVERED["channels"].add(_channels(images, labels))


# ---- b. source layouts x frame counts -----------------------------------------------------------------

# mcs_launch_weighted takes the word path only when every camera's base address, row pitch and frame
# stride (the stride counts only when F > 1) are multiples of 4 bytes; otherwise every camera is read
# with byte loads.
#   aligned      every base, pitch and frame stride a multiple of 4               -> word path
#   odd_base     aligned pitches and frame strides, base offsets of 1-3 bytes     -> byte path
#   odd_pitch    one camera's row pitch is not a multiple of 4                     -> byte path
#   odd_fstride  aligned bases and pitches, one camera's frame stride odd (F > 1)  -> byte path
# Within the word path each pixel still takes byte loads where a tap leaves the frame or the row below
# the taps would (sy + 2 >= src_h).
LAYOUTS = [(1, "aligned"), (4, "odd_base"), (11, "odd_pitch"), (13, "odd_fstride"), (19, "aligned"),
           (21, "odd_pitch"), (27, "odd_base"), (3, "odd_fstride"), (14, "aligned"), (0, "odd_pitch")]
FRAME_COUNTS = (1, 15, 16, 17, 32, 33)


def _layout(rng, layout, n_cams, row_bytes, h, F):
    """Per camera ``(offset, pitch, frame_stride)`` of a source buffer for ``layout``."""
    out = []
    odd_cam = int(rng.integers(0, n_cams))
    for k in range(n_cams):
        pitch = row_bytes + (-row_bytes) % 4 + 4 * int(rng.integers(0, 2))   # 0-7 bytes of pad, a multiple of 4
        off = 4 * int(rng.integers(0, 2))
        fpad = 4 * int(rng.integers(0, 3))
        if layout == "odd_base":
            off = int(rng.integers(0, 4)) if k != odd_cam else int(rng.integers(1, 4))
        elif layout == "odd_pitch" and k == odd_cam:
            pitch = row_bytes + int(rng.integers(0, 8))
            if pitch % 4 == 0:
                pitch += 1
        elif layout == "odd_fstride" and k == odd_cam:
            fpad += int(rng.integers(1, 4))
        out.append((off, pitch, h * pitch + fpad))
    return out


@pytest.mark.parametrize("seed,layout", LAYOUTS)
def test_source_layouts_and_frame_counts_on_random_rigs(cuda_device, seed, layout):
    import torch
    st, states, labels, images = _rig(seed)
    rng = np.random.default_rng(7005 + seed)
    F = int(rng.choice(FRAME_COUNTS if layout != "odd_fstride" else FRAME_COUNTS[1:]))
    C = _channels(images, labels)
    maps = make_maps(images, labels, MAP_KINDS[(seed + 3) % len(MAP_KINDS)], seed=seed + 50)
    st.camera_weights = maps
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    sets = [{l: rng.integers(0, 256, size=images[l].shape, dtype=np.uint8) for l in labels} for _ in range(F)]
    h, w = images[labels[0]].shape[:2]   # the cameras of a random rig share one frame size
    frames, words = [], True
    for l, (off, pitch, fstride) in zip(labels, _layout(rng, layout, len(labels), w * C, h, F)):
        buf = torch.full((off + F * fstride + 16,), 0x5A, dtype=torch.uint8, device=cuda_device)
        assert buf.data_ptr() % 16 == 0
        shape, strides = ((F, h, w, C), (fstride, pitch, C, 1)) if C > 1 else ((F, h, w), (fstride, pitch, 1))
        view = torch.as_strided(buf, shape, strides, off)
        view.copy_(torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device))
        frames.append(view)
        words = words and (view.data_ptr() | pitch | (fstride if F > 1 else 0)) % 4 == 0
    assert words == (layout == "aligned")
    row = plan.out_w * C
    opitch = row + int(rng.integers(1, 40))
    ofstride = plan.out_h * opitch + int(rng.integers(1, 64))
    poison = torch.full((F * ofstride + 64,), 0xAB, dtype=torch.uint8, device=cuda_device)
    oshape, ostrides = (((F, plan.out_h, plan.out_w, C), (ofstride, opitch, C, 1)) if C > 1 else
                        ((F, plan.out_h, plan.out_w), (ofstride, opitch, 1)))
    out = torch.as_strided(poison, oshape, ostrides)
    plan.run(frames, out=out, n_frames=F)
    assert plan.handle.last_variant() == 5
    got = out.cpu().numpy()
    for f in range(F):
        assert np.array_equal(got[f], layer_model(st, labels, sets[f], maps)[0]), f
    written = np.zeros(poison.numel(), bool)
    written[np.lib.stride_tricks.as_strided(np.arange(poison.numel()), oshape,
                                            [s * 8 for s in ostrides]).ravel()] = True
    assert bool((poison.cpu().numpy()[~written] == 0xAB).all())
    COVERED["paths"].add("word" if words else "byte")
    COVERED["frames"].add(F)


# ---- c. the contributor limit --------------------------------------------------------------------------

def _plan(flat, device):
    from multicamera_stitching_b200.engine import CompiledPlan
    return CompiledPlan(flat, device)


def _check_refused(plan, flat, frames, maps, device):
    """``maps`` put more than 4 contributors on a pixel: the setter refuses them and the plan stays in the
    overwrite, which equals the composite model."""
    import torch
    with pytest.raises(_cabi.McsError, match="code -3"):
        plan.handle.set_camera_weights(maps)
    assert not plan.handle.camera_weighted
    got = plan.run(_dev(torch, frames, device)).cpu().numpy()
    assert plan.handle.last_variant() in (1, 2)
    ref, _ = composite_model.composite(flat.layers, flat.out_w, flat.out_h, frames)
    assert np.array_equal(got, ref)


def _limit_rig(seed):
    """A COPY layer and 4-7 near-identity WARP layers over a 150 x 90 panorama, with weight maps that are zero
    outside a random vertical band of each camera (and on 10 % of the pixels inside it): how many bands
    overlap decides whether the most contributors are 4 or 5 or more.  Returns (flat, frames, maps)."""
    rng = np.random.default_rng(4000 + seed)
    C = int(rng.choice([1, 3, 4]))
    W, H = 150, 90
    layers = [Layer(0, LAYER_COPY, None, 3, 2, (3, 2, 143, 86), (84, 140))]
    for k in range(1, 1 + int(rng.integers(4, 8))):
        a = np.radians(rng.uniform(-3, 3))
        s = rng.uniform(0.95, 1.05)
        Hk = np.array([[s * np.cos(a), -s * np.sin(a), rng.uniform(-4, 4)],
                       [s * np.sin(a), s * np.cos(a), rng.uniform(-4, 4)],
                       [rng.uniform(-1e-4, 1e-4), rng.uniform(-1e-4, 1e-4), 1.0]])
        layers.append(Layer(k, LAYER_WARP, Hk, 0, 0, (0, 0, W, H), (int(rng.integers(84, 96)), int(rng.integers(140, 156)))))
    frames, maps = [], []
    for l in layers:
        h, w = l.src_hw
        frames.append(rng.integers(0, 256, size=(h, w) if C == 1 else (h, w, C), dtype=np.uint8))
        m = rng.integers(1, 256, size=(h, w), dtype=np.uint8)
        m[rng.random((h, w)) < 0.1] = 0
        band = int(rng.integers(w // 4, w // 2))
        x0 = int(rng.integers(0, w - band))
        m[:, :x0] = 0
        m[:, x0 + band:] = 0
        maps.append(m)
    return FlatPlan(layers, W, H, C, 2 if C == 1 else 3), frames, maps


LIMIT_SEEDS = range(10)


@pytest.mark.parametrize("seed", LIMIT_SEEDS)
def test_contributor_limit_on_random_overlaps(cuda_device, seed):
    flat, frames, maps = _limit_rig(seed)
    most = _blend(flat, frames, maps)[2]
    plan = _plan(flat, cuda_device)
    if most > MAX:
        _check_refused(plan, flat, frames, maps, cuda_device)
        return
    plan.handle.set_camera_weights(maps)
    assert plan.handle.camera_weighted
    _check_accepted(plan, flat, frames, maps, cuda_device)
    if most == MAX:
        COVERED["accepted_most4"] += 1


# output 135 x 53: neither a multiple of the counter's 32 x 16 blocks
ISO_W, ISO_H = 135, 53
ISO_SPOTS = {"lane31": (63, 20), "last_row_and_column": (ISO_W - 1, ISO_H - 1), "interior": (70, 30), "origin": (0, 0)}


def _isolated_rig(spot, base, most):
    """A COPY layer and four integer-translation WARP layers (every tap at ax = ay = 0, so a weight is exactly the
    map byte under it).  The first ``base`` layers have maps of 1..255 everywhere; the others have maps that are
    zero except one 255 byte that lands on output pixel ``spot``.  ``most == 5`` puts every spot there;
    ``most == 4`` moves the last one to a neighbouring pixel.  Returns (flat, frames, maps)."""
    rng = np.random.default_rng(100 * base + most)
    layers = [Layer(0, LAYER_COPY, None, 0, 0, (0, 0, ISO_W, ISO_H), (ISO_H, ISO_W))]
    shifts = [(0, 0)]
    for k in range(1, 5):
        tx, ty = int(rng.integers(-5, 1)), int(rng.integers(-5, 1))
        Hk = np.array([[1.0, 0, tx], [0, 1.0, ty], [0, 0, 1.0]])
        layers.append(Layer(k, LAYER_WARP, Hk, 0, 0, (0, 0, ISO_W, ISO_H), (ISO_H + 5, ISO_W + 5)))
        shifts.append((tx, ty))
    frames, maps = [], []
    for k, l in enumerate(layers):
        h, w = l.src_hw
        frames.append(rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8))
        if k < base:
            maps.append(rng.integers(1, 256, size=(h, w), dtype=np.uint8))
            continue
        x, y = spot
        if most == 4 and k == 4:
            x = x - 1 if x > 0 else x + 1
        m = np.zeros((h, w), np.uint8)
        m[y - shifts[k][1], x - shifts[k][0]] = 255
        maps.append(m)
    return FlatPlan(layers, ISO_W, ISO_H, 3, 3), frames, maps


@pytest.mark.parametrize("most", [5, 4])
@pytest.mark.parametrize("base", [0, 3])
@pytest.mark.parametrize("spot", list(ISO_SPOTS))
def test_contributor_limit_at_one_isolated_pixel(cuda_device, spot, base, most):
    flat, frames, maps = _isolated_rig(ISO_SPOTS[spot], base, most)
    _, contrib, m = _blend(flat, frames, maps)
    assert m == most
    if base == 0:
        assert contrib == [1] * 5
    plan = _plan(flat, cuda_device)
    if most > MAX:
        _check_refused(plan, flat, frames, maps, cuda_device)
        COVERED["refused_isolated5"] += 1
        return
    plan.handle.set_camera_weights(maps)
    _check_accepted(plan, flat, frames, maps, cuda_device)
    COVERED["accepted_most4"] += 1


# ---- d. divisors at both ends --------------------------------------------------------------------------

def _stack(n, w, half=False, c=3, h=64, seed=0):
    """``n`` cameras over the middle of a 128 x 80 panorama: a COPY layer at (8, 8) and WARP layers with small
    shifts, shears and scales, or (``half``) translations by whole and half pixels, so that weights and values
    are means of two or four taps.  Returns (flat, frames)."""
    rng = np.random.default_rng(seed)
    layers = [Layer(0, LAYER_COPY, None, 8, 8, (8, 8, 8 + w, 8 + h), (h, w))]
    for k in range(1, n):
        if half:
            H = np.array([[1.0, 0, 4 * k + 0.5 * (k & 1)], [0, 1.0, 2 * k + 0.5 * (k >> 1 & 1)], [0, 0, 1]])
        else:
            H = np.array([[1 + 0.02 * k, 0.01 * k, 4 * k], [0.005 * k, 1 - 0.01 * k, 3 * k], [1e-5 * k, 0, 1]])
        layers.append(Layer(k, LAYER_WARP, H, 0, 0, (0, 0, 128, 80), (h, w)))
    frames = [rng.integers(0, 256, size=(h, w, c), dtype=np.uint8) for _ in range(n)]
    return FlatPlan(layers, 128, 80, c, 3), frames


DIVISOR_MAPS = ("ones", "ones_and_twos", "full", "random")


def _divisor_maps(kind, shapes, seed):
    rng = np.random.default_rng(seed)
    if kind == "ones":              # S = the number of contributors, 2..4
        return [np.ones(s, np.uint8) for s in shapes]
    if kind == "ones_and_twos":
        return [rng.integers(1, 3, size=s, dtype=np.uint8) for s in shapes]
    if kind == "full":              # S up to 4 * 255
        return [np.full(s, 255, np.uint8) for s in shapes]
    return [rng.integers(0, 256, size=s, dtype=np.uint8) for s in shapes]


@pytest.mark.parametrize("kind", DIVISOR_MAPS)
@pytest.mark.parametrize("stack", ["warps_word", "half_pixel_word", "half_pixel_byte"])
def test_divisors_on_a_four_deep_stack(cuda_device, stack, kind):
    # 96 x 3 bytes per row: the word path; 97 x 3: the byte path
    flat, frames = _stack(4, 97 if stack.endswith("byte") else 96, half=stack.startswith("half"), seed=len(kind))
    maps = _divisor_maps(kind, [f.shape[:2] for f in frames], seed=11)
    plan = _plan(flat, cuda_device)
    plan.handle.set_camera_weights(maps)
    assert _check_accepted(plan, flat, frames, maps, cuda_device) == 4


@pytest.mark.parametrize("kind", DIVISOR_MAPS[:3])
@pytest.mark.parametrize("seed", [1, 20])
def test_divisors_on_random_rigs(cuda_device, seed, kind):
    st, states, labels, images = _rig(seed)
    maps = dict(zip(labels, _divisor_maps(kind, [images[l].shape[:2] for l in labels], seed)))
    ref, contrib, most = layer_model(st, labels, images, maps)
    assert most == MAX
    st.camera_weights = maps
    assert np.array_equal(st.stitch(images), ref)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.last_variant() == 5 and plan.owned_pixels() == contrib


# ---- e. REMAP layers -----------------------------------------------------------------------------------

def _remap_rig(seed):
    """2-4 layers over a 200 x 120 panorama: a COPY layer, then WARP and REMAP layers; the REMAP layers
    undistort with random coefficients or follow random fixed-point maps whose taps leave the source."""
    rng = np.random.default_rng(9000 + seed)
    W, H, C = 200, 120, int(rng.choice([1, 3, 4]))
    layers = [Layer(0, LAYER_COPY, None, 20, 10, (20, 10, 180, 100), (90, 160))]
    for k in range(1, int(rng.integers(2, 5))):
        what = ("warp", "undistort", "random_map")[(seed + k) % 3]
        if what == "warp":
            Hk = np.array([[1 + rng.uniform(-0.05, 0.05), rng.uniform(-0.03, 0.03), rng.uniform(0, 40)],
                           [rng.uniform(-0.03, 0.03), 1 + rng.uniform(-0.05, 0.05), rng.uniform(0, 20)],
                           [rng.uniform(-1e-4, 1e-4), 0, 1]])
            layers.append(Layer(k, LAYER_WARP, Hk, 0, 0, (0, 0, W, H), (100, 170)))
        elif what == "undistort":
            A = np.array([[rng.uniform(150, 250), 0, W / 2 + rng.uniform(-5, 5)],
                          [0, rng.uniform(150, 250), H / 2 + rng.uniform(-5, 5)], [0, 0, 1]])
            dist = np.array([rng.uniform(-0.35, 0.1), rng.uniform(-0.05, 0.15), rng.uniform(-3e-3, 3e-3),
                             rng.uniform(-3e-3, 3e-3), 0.0])
            xy, frac = prewarp.undistort_maps(A, dist, (W, H))
            layers.append(Layer(k, LAYER_REMAP, None, 0, 0, (0, 0, W, H), (H, W), (xy, frac)))
        else:
            ys, xs = np.mgrid[0:H, 0:W]
            xy = np.stack([xs - 30 + rng.integers(-1, 2, size=xs.shape), ys - 12 + rng.integers(-1, 2, size=xs.shape)],
                          axis=-1).astype(np.int16)
            frac = rng.integers(0, 1024, size=xs.shape).astype(np.uint16)
            layers.append(Layer(k, LAYER_REMAP, None, 0, 0, (0, 0, W, H), (96, 150), (xy, frac)))
    frames = [rng.integers(0, 256, size=l.src_hw if C == 1 else tuple(l.src_hw) + (C,), dtype=np.uint8)
              for l in layers]
    maps = make_maps({k: f for k, f in enumerate(frames)}, range(len(frames)), MAP_KINDS[seed % len(MAP_KINDS)],
                     seed=seed)
    return FlatPlan(layers, W, H, C, 2 if C == 1 else 3), frames, [maps[k] for k in range(len(frames))]


@pytest.mark.parametrize("seed", range(8))
def test_remap_layers_with_random_maps(cuda_device, seed):
    flat, frames, maps = _remap_rig(seed)
    plan = _plan(flat, cuda_device)
    plan.handle.set_camera_weights(maps)
    _check_accepted(plan, flat, frames, maps, cuda_device)


# ---- f. the map pitch of the C ABI ---------------------------------------------------------------------

def test_map_pitch_of_the_c_abi(cuda_device):
    """mcs_plan_set_camera_weights copies each map row by row with its own pitch: maps handed over as
    windows of wider arrays, whose padding would change the panorama if it were read, give what the
    contiguous maps give."""
    import torch
    flat, frames = _stack(4, 97, seed=3)
    rng = np.random.default_rng(3)
    maps = [rng.integers(1, 256, size=f.shape[:2], dtype=np.uint8) for f in frames]
    maps[2] = None
    plan = _plan(flat, cuda_device)
    plan.handle.set_camera_weights(maps)
    want = plan.run(_dev(torch, frames, cuda_device)).cpu().numpy()
    owned = plan.owned_pixels()
    assert np.array_equal(want, _blend(flat, frames, maps)[0])
    n = len(maps)
    ptrs = (ctypes.c_void_p * n)()
    pitches = np.zeros(n, np.int64)
    wide = []
    for k, m in enumerate(maps):
        if m is None:
            continue
        h, w = m.shape
        big = np.zeros((h, w + 1 + 6 * k), np.uint8)   # pads of 1, 7 and 19 bytes, all weight 0
        big[:, :w] = m
        # read as if the rows were contiguous, these maps would give another panorama
        assert not np.array_equal(_blend(flat, frames, [big.ravel()[:h * w].reshape(h, w) if j == k else mm
                                                        for j, mm in enumerate(maps)])[0], want)
        wide.append(big)
        ptrs[k] = big.ctypes.data
        pitches[k] = big.strides[0]
    rc = _cabi.load().mcs_plan_set_camera_weights(plan.handle._h, ptrs,
                                                  pitches.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))
    assert rc == 0, _cabi.load().mcs_last_error().decode()
    plan.handle._owned = None
    got = plan.run(_dev(torch, frames, cuda_device)).cpu().numpy()
    assert plan.handle.last_variant() == 5
    assert np.array_equal(got, want)
    assert plan.owned_pixels() == owned


# ---- g. what the file exercised ------------------------------------------------------------------------

def test_fuzz_exercised_the_camera_weight_space(cuda_device):
    assert len(COVERED["rigs_3plus"]) >= 5, COVERED
    assert COVERED["mirrored"], COVERED
    assert COVERED["channels"] >= {1, 3, 4}, COVERED
    assert COVERED["paths"] == {"word", "byte"}, COVERED
    F = COVERED["frames"]
    assert min(F) <= 16 < max(F) and any(f <= 32 for f in F) and any(f > 32 for f in F), COVERED
    assert any(f < 16 for f in F) and any(16 < f <= 32 for f in F), COVERED
    assert COVERED["accepted_most4"] >= 1 and COVERED["refused_isolated5"] >= 1, COVERED
