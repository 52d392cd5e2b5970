"""Voronoi seams of the multi-band blend on the GPU (csrc/mcs_seams.cu): every comparison is ``np.array_equal``
against ``oracle/seam_model.find`` (the seam-cut weights, read back per layer) and ``oracle/seam_model.blend``
(the panorama; ``oracle/multiband_model.blend`` where the seams are off) on the plan's own flattening.

- the seeded random rigs under the map kinds, numpy frames and device frames;
- frame counts around the 16-frame workspace sub-batch, and SequencePipeline;
- switching the seams off gives back the blend without them, and the calls that switch them off;
- the C ABI's error paths, including the W + H refusal on a synthetic wide plan;
- a mask whose only unique pixels lie exactly 10 pixels beyond the overlap (the submask's gap);
- one full-size config-2 frame-set at 5 bands against cv2's VoronoiSeamFinder and MultiBandBlender directly."""
import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, chain_case, make_maps
from multicamera_stitching_b200 import _cabi, edge_ramp
from multicamera_stitching_b200.plan import LAYER_COPY, LAYER_WARP, FlatPlan, Layer, PlanUnsupported, flatten_chain
from oracle import multiband_model, seam_model
from random_rigs import random_chain

pytestmark = pytest.mark.gpu

COVERED = {"rigs": set(), "kinds": set(), "bands": set(), "channels": set(), "frames": set(), "layers": 0,
           "sequence": 0, "cv2_full": 0, "off": 0, "errors": 0, "bound": 0, "gap": 0}


def _flat(st, labels, images):
    return flatten_chain(st.stitchers, [images[l].shape for l in labels])


def _model(st, labels, images, maps, bands, seams=True):
    flat = _flat(st, labels, images)
    blend = seam_model.blend if seams else multiband_model.blend
    return blend(flat.layers, flat.out_w, flat.out_h, [images[l] for l in labels], [maps.get(l) for l in labels], bands)


def _expected_seams(flat, frames, maps, finder=seam_model.find):
    """``{layer index: seam-cut weights}`` of the layers that feed the blend."""
    fed = []
    for k, l in enumerate(flat.layers):
        x0, y0, x1, y1 = [int(v) for v in l.rect]
        if min(flat.out_w, x1) > max(0, x0) and min(flat.out_h, y1) > max(0, y0):
            fed.append(k)
    planes = multiband_model.camera_planes(flat.layers, flat.out_w, flat.out_h, frames, maps)
    assert len(planes) == len(fed)
    return dict(zip(fed, finder(*seam_model.plane_inputs(planes))))


def _check_seams(handle, flat, frames, maps, finder=seam_model.find):
    want = _expected_seams(flat, frames, maps, finder)
    for k in range(len(flat.layers)):
        if k in want:
            got = handle.seam_weights(k)
            assert got.shape == want[k].shape and np.array_equal(got, want[k]), (k, int((got != want[k]).sum()))
            COVERED["layers"] += 1
        else:
            with pytest.raises(_cabi.McsError, match="code -1"):
                handle.seam_weights(k)


@pytest.mark.parametrize("seed", range(28))
def test_random_rig_matches_the_specification(cuda_device, seed):
    import torch
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    for i, kind in enumerate(MAP_KINDS[seed % 4::4]):
        bands = 1 + (seed + i) % 6
        maps = make_maps(images, labels, kind, seed=seed)
        st.camera_weights, st.blend_bands, st.voronoi_seams = maps, bands, True
        plan = st.plan([images[l].shape for l in labels], cuda_device)
        assert plan.handle.voronoi_seams
        _check_seams(plan.handle, plan.flat, [images[l] for l in labels], [maps.get(l) for l in labels])
        ref = _model(st, labels, images, maps, bands)
        got = st.stitch(images)
        assert got.shape == ref.shape and np.array_equal(got, ref), (kind, bands)
        dev = st.stitch({l: torch.from_numpy(images[l]).to(cuda_device) for l in labels}).cpu().numpy()
        assert np.array_equal(dev, ref), (kind, bands)
        assert plan.handle.last_variant() == 6
        COVERED["kinds"].add(kind)
        COVERED["bands"].add(bands)
    COVERED["rigs"].add(seed)
    COVERED["channels"].add(1 if images[labels[0]].ndim == 2 else images[labels[0]].shape[2])


@pytest.mark.parametrize("F", [1, 16, 17, 64])
def test_frame_counts_around_the_sub_batch(cuda_device, F):
    import torch
    st, states, labels, images = chain_case(3, 48, 80, 3)
    maps = make_maps(images, labels, "mixed", seed=F)
    st.camera_weights, st.blend_bands, st.voronoi_seams = maps, 4, True
    sets = [chain_case(3, 48, 80, 3, frame_index=f)[3] for f in range(F)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    out = st.stitch_batch(batch).cpu().numpy()
    for f in range(F):
        assert np.array_equal(out[f], _model(st, labels, sets[f], maps, 4)), f
    COVERED["frames"].add(F)


def test_sequence_pipeline(cuda_device):
    import torch
    from multicamera_stitching_b200.sequence import SequencePipeline
    st, states, labels, images = chain_case(4, 90, 160, 3)
    st.camera_weights = {l: edge_ramp(images[l].shape, 24) for l in labels}
    st.blend_bands, st.voronoi_seams = 5, True
    F = 7
    sets = [chain_case(4, 90, 160, 3, frame_index=f)[3] for f in range(F)]
    pipe = SequencePipeline(st, [images[l].shape for l in labels], cuda_device, chunk=3, depth=2)
    assert pipe.plan.handle.voronoi_seams
    host = {l: torch.from_numpy(np.stack([s[l] for s in sets])).pin_memory() for l in labels}
    ref0 = _model(st, labels, images, st.camera_weights, 5)
    out = torch.full((F,) + ref0.shape, 0xEE, dtype=torch.uint8).pin_memory()
    assert pipe.run(host, out) == F
    for f in range(F):
        assert np.array_equal(out[f].numpy(), _model(st, labels, sets[f], st.camera_weights, 5)), f
    COVERED["sequence"] += 1


@pytest.mark.parametrize("c", [1, 3, 4])
def test_switching_the_seams_off_gives_back_the_blend_without_them(cuda_device, c):
    import torch
    st, states, labels, images = chain_case(4, 72, 120, c)
    maps = make_maps(images, labels, "ramp", seed=c)
    st.camera_weights, st.blend_bands = maps, 3
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    dev = [torch.from_numpy(images[l]).to(cuda_device) for l in labels]
    without = plan.run(dev).cpu().numpy()
    assert np.array_equal(without, _model(st, labels, images, maps, 3, seams=False))
    plan.handle.set_voronoi_seams(True)
    seams = _model(st, labels, images, maps, 3)
    assert not np.array_equal(seams, without)
    assert np.array_equal(plan.run(dev).cpu().numpy(), seams)
    plan.handle.set_voronoi_seams(True)   # again: the same seams
    assert np.array_equal(plan.run(dev).cpu().numpy(), seams)
    plan.handle.set_voronoi_seams(False)
    assert not plan.handle.voronoi_seams and plan.handle.blend_bands == 3
    assert np.array_equal(plan.run(dev).cpu().numpy(), without)
    plan.handle.set_voronoi_seams(False)  # off twice
    assert np.array_equal(plan.run(dev).cpu().numpy(), without)
    COVERED["off"] += 1
    COVERED["channels"].add(c)


def _stack(cuda_device, n_layers, h=64, w=96, c=3, empty_layer=False):
    """Every camera sees the middle of a 128 x 80 panorama; optionally one more layer outside it."""
    from multicamera_stitching_b200 import synthetic
    from multicamera_stitching_b200.engine import CompiledPlan
    layers = [Layer(0, LAYER_COPY, None, 8, 8, (8, 8, 8 + w, 8 + h), (h, w))]
    for k in range(1, n_layers):
        H = np.array([[1 + 0.02 * k, 0.01 * k, 4 * k], [0.005 * k, 1 - 0.01 * k, 3 * k], [1e-5 * k, 0, 1]])
        layers.append(Layer(k, LAYER_WARP, H, 0, 0, (0, 0, 128, 80), (h, w)))
    if empty_layer:
        layers.append(Layer(n_layers, LAYER_WARP, np.eye(3), 0, 0, (140, 0, 200, 80), (h, w)))
    flat = FlatPlan(layers, 128, 80, c, 3)
    frames = [synthetic.make_frame(h, w, c, cam_index=k, kind="noise") for k in range(len(layers))]
    return CompiledPlan(flat, cuda_device), flat, frames


def test_error_paths_of_the_c_abi(cuda_device):
    import torch
    plan, flat, frames = _stack(cuda_device, 4, empty_layer=True)
    h = plan.handle
    dev = [torch.from_numpy(f).to(cuda_device) for f in frames]
    with pytest.raises(_cabi.McsError, match="code -1"):   # no multi-band blend
        h.set_voronoi_seams(True)
    maps = [edge_ramp(f.shape, 7 + k) for k, f in enumerate(frames)]
    h.set_camera_weights(maps)
    with pytest.raises(_cabi.McsError, match="code -1"):   # the single-band blend takes no seams
        h.set_voronoi_seams(True)
    h.set_multiband(4)
    with pytest.raises(_cabi.McsError, match="code -1"):   # seams off: nothing to read back
        h.seam_weights(0)
    h.set_voronoi_seams(True)
    _check_seams(h, flat, frames, maps)                   # the last layer feeds nothing: code -1
    for bad in (-1, len(flat.layers), 99):
        with pytest.raises(_cabi.McsError, match="code -1"):
            h.seam_weights(bad)
    args = (flat.layers, flat.out_w, flat.out_h, frames, maps, 4)
    assert np.array_equal(plan.run(dev).cpu().numpy(), seam_model.blend(*args))
    for v in (1, 2):
        h.force_variant(v)
        with pytest.raises(_cabi.McsError, match="code -3"):
            plan.run(dev)
    h.force_variant(0)
    # set_multiband switches the seams off
    h.set_multiband(4)
    assert not h.voronoi_seams
    with pytest.raises(_cabi.McsError, match="code -1"):
        h.seam_weights(0)
    assert np.array_equal(plan.run(dev).cpu().numpy(), multiband_model.blend(*args))
    # so does set_camera_weights, and the multi-band blend with them
    h.set_voronoi_seams(True)
    h.set_camera_weights(maps)
    assert not h.voronoi_seams and not h.multiband
    with pytest.raises(_cabi.McsError, match="code -1"):
        h.seam_weights(1)
    with pytest.raises(_cabi.McsError, match="code -1"):
        h.set_voronoi_seams(True)
    h.set_multiband(4)
    assert np.array_equal(plan.run(dev).cpu().numpy(), multiband_model.blend(*args))
    COVERED["errors"] += 1


def test_the_bound_is_refused_on_a_wide_plan(cuda_device):
    """Two cameras overlapping over a 32 760-pixel-wide panorama: the submask's W + H reaches 32 768."""
    import torch
    from multicamera_stitching_b200 import synthetic
    from multicamera_stitching_b200.engine import CompiledPlan
    out_w, out_h = 32760, 4
    layers = [Layer(k, LAYER_WARP, np.array([[1.0, 0, -3 * k], [0, 1, 0], [0, 0, 1]]), 0, 0, (0, 0, out_w, out_h),
                    (16, 16)) for k in range(2)]
    flat = FlatPlan(layers, out_w, out_h, 3, 3)
    assert not seam_model.supported([(out_w, out_h)] * 2, [(0, 0)] * 2)
    frames = [synthetic.make_frame(16, 16, 3, cam_index=k, kind="noise") for k in range(2)]
    dev = [torch.from_numpy(f).to(cuda_device) for f in frames]
    plan = CompiledPlan(flat, cuda_device, camera_weights=[None, None], blend_bands=2)
    before = plan.run(dev).cpu().numpy()
    with pytest.raises(_cabi.McsError, match="code -3"):
        plan.handle.set_voronoi_seams(True)
    assert not plan.handle.voronoi_seams and plan.handle.multiband
    with pytest.raises(_cabi.McsError, match="code -1"):
        plan.handle.seam_weights(0)
    assert np.array_equal(plan.run(dev).cpu().numpy(), before)   # the plan stayed as it was
    assert np.array_equal(before, multiband_model.blend(flat.layers, out_w, out_h, frames, [None, None], 2))
    with pytest.raises(PlanUnsupported, match="32768"):
        CompiledPlan(flat, cuda_device, camera_weights=[None, None], blend_bands=2, voronoi_seams=True)
    COVERED["bound"] += 1


@pytest.mark.parametrize("col", [10, 9])
def test_the_submask_reaches_ten_pixels_beyond_the_overlap(cuda_device, col):
    """Two pasted cameras overlapping in columns 20-39; camera 0's only unique pixels are column ``col``: at 10
    pixels from the overlap they win its left quarter, at 11 they are outside every submask."""
    import torch
    from multicamera_stitching_b200 import synthetic
    from multicamera_stitching_b200.engine import CompiledPlan
    layers = [Layer(0, LAYER_COPY, None, 0, 0, (0, 0, 40, 20), (20, 40)),
              Layer(1, LAYER_COPY, None, 20, 0, (20, 0, 60, 20), (20, 40))]
    flat = FlatPlan(layers, 60, 20, 3, 3)
    m0 = np.zeros((20, 40), np.uint8)
    m0[:, col] = 255
    m0[:, 20:] = 200
    maps = [m0, np.full((20, 40), 255, np.uint8)]
    frames = [synthetic.make_frame(20, 40, 3, cam_index=k, kind="noise") for k in range(2)]
    plan = CompiledPlan(flat, cuda_device, camera_weights=maps, blend_bands=3, voronoi_seams=True)
    _check_seams(plan.handle, flat, frames, maps)
    assert list(np.nonzero(plan.handle.seam_weights(0)[0])[0]) == ([10, 20, 21, 22, 23, 24] if col == 10 else [9])
    got = plan.run([torch.from_numpy(f).to(cuda_device) for f in frames]).cpu().numpy()
    assert np.array_equal(got, seam_model.blend(flat.layers, 60, 20, frames, maps, 3))
    COVERED["gap"] += 1


def test_full_size_config2_against_cv2(cuda_device):
    from multicamera_stitching_b200 import synthetic
    n, h, w = synthetic.CONFIGS["cfg2_6x1080p"]
    st, _, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, kind="smooth")
    maps = {l: edge_ramp(images[l].shape, 64) for l in labels}
    st.camera_weights, st.blend_bands, st.voronoi_seams = maps, 5, True
    plan = st.plan([images[l].shape for l in labels])
    flat = plan.flat
    frames, m = [images[l] for l in labels], [maps[l] for l in labels]
    _check_seams(plan.handle, flat, frames, m, seam_model.find_cv2)
    got = st.stitch(images)
    ref = seam_model.blend_cv2(flat.layers, flat.out_w, flat.out_h, frames, m, 5)
    assert np.array_equal(got, ref), int(np.abs(got.astype(int) - ref.astype(int)).max())
    COVERED["cv2_full"] += 1


def test_the_file_reached_what_it_claims():
    assert len(COVERED["rigs"]) >= 20, COVERED["rigs"]
    assert COVERED["kinds"] == set(MAP_KINDS), COVERED["kinds"]
    assert COVERED["bands"] == set(range(1, 7)), COVERED["bands"]
    assert COVERED["channels"] == {1, 3, 4}
    assert COVERED["frames"] == {1, 16, 17, 64}
    assert COVERED["layers"] >= 60, COVERED["layers"]
    assert COVERED["sequence"] == 1 and COVERED["cv2_full"] == 1 and COVERED["off"] == 3
    assert COVERED["errors"] == 1 and COVERED["bound"] == 1 and COVERED["gap"] == 2
