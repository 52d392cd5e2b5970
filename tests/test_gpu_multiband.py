"""Multi-band blend on the GPU (csrc/mcs_stitch_multiband.cu, variant 6): every comparison is
``np.array_equal`` against ``oracle/multiband_model.blend`` on the plan's own flattening.

- the seeded random rigs and synthetic chains under every map kind, 1-6 bands, numpy frames and device batches;
- frame counts around the 16-frame workspace sub-batch;
- poisoned, padded outputs and strided or unaligned sources;
- rigs where more than 4 cameras cover one pixel (the camera-weighted kernel refuses them);
- SequencePipeline with poisoned slots;
- the C ABI's error paths and the way back to the single-band blend;
- one full-size config-2 frame-set at 5 bands against cv2's MultiBandBlender directly."""
import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, chain_case, make_maps
from multicamera_stitching_b200 import _cabi, edge_ramp
from multicamera_stitching_b200.plan import LAYER_COPY, LAYER_WARP, FlatPlan, Layer, flatten_chain
from oracle import camera_weight_model, composite_model, multiband_model
from random_rigs import random_chain

pytestmark = pytest.mark.gpu

COVERED = {"rigs": set(), "bands": set(), "channels": set(), "frames": set(), "most_over_4": 0, "layouts": set(),
           "sequence": 0, "cv2_full": 0}


def _model(st, labels, images, maps, bands):
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    return multiband_model.blend(flat.layers, flat.out_w, flat.out_h, [images[l] for l in labels],
                                 [maps.get(l) for l in labels], bands)


def _diff(a, b):
    return int(np.abs(a.astype(int) - b.astype(int)).max())


@pytest.mark.parametrize("seed", range(28))
def test_random_rig_matches_the_specification(cuda_device, seed):
    import torch
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    for i, kind in enumerate(MAP_KINDS[seed % 3::3]):
        bands = 1 + (seed + i) % 6
        maps = make_maps(images, labels, kind, seed=seed)
        st.camera_weights, st.blend_bands = maps, bands
        ref = _model(st, labels, images, maps, bands)
        got = st.stitch(images)
        assert got.shape == ref.shape and np.array_equal(got, ref), (kind, bands, _diff(got, ref))
        dev = st.stitch({l: torch.from_numpy(images[l]).to(cuda_device) for l in labels}).cpu().numpy()
        assert np.array_equal(dev, ref), (kind, bands)
        plan = st.plan([images[l].shape for l in labels], cuda_device)
        assert plan.handle.last_variant() == 6
        flat = plan.flat
        assert plan.handle.blend_bands == multiband_model.num_bands(bands, flat.out_w, flat.out_h)
        assert all(win == (0, 0, int(l.src_hw[1]), int(l.src_hw[0]))
                   for win, l in zip(plan.handle.source_windows(), flat.layers))
        COVERED["bands"].add(bands)
    COVERED["rigs"].add(seed)
    COVERED["channels"].add(1 if images[labels[0]].ndim == 2 else images[labels[0]].shape[2])


@pytest.mark.parametrize("c,bands", [(1, 2), (3, 5), (4, 3)])
def test_without_maps_every_camera_weighs_255(cuda_device, c, bands):
    st, states, labels, images = chain_case(4, 72, 120, c)
    st.blend_bands = bands
    got = st.stitch(images)
    assert np.array_equal(got, _model(st, labels, images, {}, bands))
    COVERED["channels"].add(c)


@pytest.mark.parametrize("F", [1, 15, 16, 17, 33, 64])
def test_frame_counts_around_the_sub_batch(cuda_device, F):
    import torch
    st, states, labels, images = chain_case(3, 48, 80, 3)
    maps = make_maps(images, labels, "mixed", seed=F)
    st.camera_weights, st.blend_bands = maps, 4
    sets = [chain_case(3, 48, 80, 3, frame_index=f)[3] for f in range(F)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    out = st.stitch_batch(batch).cpu().numpy()
    for f in range(F):
        assert np.array_equal(out[f], _model(st, labels, sets[f], maps, 4)), f
    COVERED["frames"].add(F)


def _strided(torch, arr, pitch, offset, device):
    F, h = arr.shape[0], arr.shape[1]
    buf = torch.zeros(offset + F * h * pitch + 16, dtype=torch.uint8, device=device)
    view = torch.as_strided(buf, arr.shape, (h * pitch, pitch, arr.shape[3], 1), offset)
    view.copy_(torch.from_numpy(arr).to(device))
    return view


@pytest.mark.parametrize("w,pitch_pad,offset,F", [(160, 0, 0, 3), (160, 4, 1, 17), (131, 3, 2, 5), (131, 0, 0, 18)])
def test_strided_sources_into_a_poisoned_padded_output(cuda_device, w, pitch_pad, offset, F):
    import torch
    st, states, labels, images = chain_case(3, 80, w, 3)
    maps = make_maps(images, labels, "random", seed=w)
    st.camera_weights, st.blend_bands = maps, 3
    sets = [chain_case(3, 80, w, 3, frame_index=f)[3] for f in range(F)]
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    frames = [_strided(torch, np.stack([s[l] for s in sets]), w * 3 + pitch_pad, offset, cuda_device) for l in labels]
    row = plan.out_w * 3
    pitch = row + 29
    poison = torch.full((F * plan.out_h * pitch + 7,), 0xAB, dtype=torch.uint8, device=cuda_device)
    out = torch.as_strided(poison, (F, plan.out_h, plan.out_w, 3), (plan.out_h * pitch, pitch, 3, 1), 3)
    plan.run(frames, out=out, n_frames=F)
    assert plan.handle.last_variant() == 6
    got = out.cpu().numpy()
    for f in range(F):
        assert np.array_equal(got[f], _model(st, labels, sets[f], maps, 3)), f
    view = poison[3:3 + F * plan.out_h * pitch].view(F, plan.out_h, pitch)
    assert bool((view[:, :, row:] == 0xAB).all()) and bool((poison[:3] == 0xAB).all())
    COVERED["layouts"].add((w, pitch_pad, offset))


def _stack(cuda_device, n_layers, h=64, w=96, c=3):
    """Every camera sees the middle of a 128 x 80 panorama."""
    from multicamera_stitching_b200 import synthetic
    from multicamera_stitching_b200.engine import CompiledPlan
    layers = [Layer(0, LAYER_COPY, None, 8, 8, (8, 8, 8 + w, 8 + h), (h, w))]
    for k in range(1, n_layers):
        H = np.array([[1 + 0.02 * k, 0.01 * k, 4 * k], [0.005 * k, 1 - 0.01 * k, 3 * k], [1e-5 * k, 0, 1]])
        layers.append(Layer(k, LAYER_WARP, H, 0, 0, (0, 0, 128, 80), (h, w)))
    flat = FlatPlan(layers, 128, 80, c, 3)
    frames = [synthetic.make_frame(h, w, c, cam_index=k, kind="noise") for k in range(n_layers)]
    return CompiledPlan(flat, cuda_device), flat, frames


@pytest.mark.parametrize("n_layers,bands", [(5, 3), (7, 5), (9, 6)])
def test_more_than_four_cameras_on_one_pixel(cuda_device, n_layers, bands):
    import torch
    plan, flat, frames = _stack(cuda_device, n_layers)
    maps = [edge_ramp(f.shape, 5 + 3 * k) for k, f in enumerate(frames)]
    assert camera_weight_model.blend(flat.layers, flat.out_w, flat.out_h, frames, maps)[2] > 4
    with pytest.raises(_cabi.McsError, match="code -3"):
        plan.handle.set_camera_weights(maps)
    dev = [torch.from_numpy(f).to(cuda_device) for f in frames]
    # refused by the camera-weighted kernel: the overwrite serves the plan
    overwrite = composite_model.composite(flat.layers, flat.out_w, flat.out_h, frames)[0]
    assert np.array_equal(plan.run(dev).cpu().numpy(), overwrite)
    plan.handle.set_multiband(bands)
    got = plan.run(dev).cpu().numpy()
    assert plan.handle.last_variant() == 6
    assert np.array_equal(got, multiband_model.blend(flat.layers, flat.out_w, flat.out_h, frames, maps, bands))
    plan.handle.set_multiband(0)
    assert np.array_equal(plan.run(dev).cpu().numpy(), overwrite)
    COVERED["most_over_4"] += 1


def test_error_paths_of_the_c_abi(cuda_device):
    import torch
    plan, flat, frames = _stack(cuda_device, 4)
    dev = [torch.from_numpy(f).to(cuda_device) for f in frames]
    with pytest.raises(_cabi.McsError, match="code -1"):   # no camera weights
        plan.handle.set_multiband(3)
    maps = [edge_ramp(f.shape, 7 + k) for k, f in enumerate(frames)]
    plan.handle.set_camera_weights(maps)
    for bad in (-1, 9, 100):
        with pytest.raises(_cabi.McsError, match="code -1"):
            plan.handle.set_multiband(bad)
    assert plan.handle.set_multiband(8) == multiband_model.num_bands(8, flat.out_w, flat.out_h) == 7
    ref = multiband_model.blend(flat.layers, flat.out_w, flat.out_h, frames, maps, 8)
    assert np.array_equal(plan.run(dev).cpu().numpy(), ref) and plan.handle.last_variant() == 6
    for v in (1, 2):
        plan.handle.force_variant(v)
        with pytest.raises(_cabi.McsError, match="code -3"):
            plan.run(dev)
    plan.handle.force_variant(0)
    with pytest.raises(_cabi.McsError, match="code -1"):   # the stage-wise blend is excluded
        plan.handle.set_feather(2)
    # back to the single-band blend
    plan.handle.set_multiband(0)
    assert plan.handle.blend_bands == 0
    cw = camera_weight_model.blend(flat.layers, flat.out_w, flat.out_h, frames, maps)[0]
    assert np.array_equal(plan.run(dev).cpu().numpy(), cw) and plan.handle.last_variant() == 5
    # new maps switch the mode off; clearing the maps clears it too
    plan.handle.set_multiband(2)
    plan.handle.set_camera_weights(None)
    assert np.array_equal(plan.run(dev).cpu().numpy(), composite_model.composite(flat.layers, flat.out_w, flat.out_h, frames)[0])
    with pytest.raises(_cabi.McsError, match="code -1"):
        plan.handle.set_multiband(2)


def test_sequence_pipeline_with_poisoned_slots(cuda_device):
    import torch
    from multicamera_stitching_b200.sequence import SequencePipeline
    st, states, labels, images = chain_case(4, 90, 160, 3)
    st.camera_weights = {l: edge_ramp(images[l].shape, 24) for l in labels}
    st.blend_bands = 5
    F = 7
    sets = [chain_case(4, 90, 160, 3, frame_index=f)[3] for f in range(F)]
    pipe = SequencePipeline(st, [images[l].shape for l in labels], cuda_device, chunk=3, depth=2)
    for slot in pipe.slots:   # poison the device slots
        for t in slot["src"]:
            t.fill_(0xCD)
        slot["dst"].fill_(0xCD)
    host = {l: torch.from_numpy(np.stack([s[l] for s in sets])).pin_memory() for l in labels}
    ref0 = _model(st, labels, images, st.camera_weights, 5)
    out = torch.full((F,) + ref0.shape, 0xEE, dtype=torch.uint8).pin_memory()
    assert pipe.run(host, out) == F
    for f in range(F):
        assert np.array_equal(out[f].numpy(), _model(st, labels, sets[f], st.camera_weights, 5)), f
    COVERED["sequence"] += 1


def test_full_size_config2_against_cv2(cuda_device):
    from multicamera_stitching_b200 import synthetic
    n, h, w = synthetic.CONFIGS["cfg2_6x1080p"]
    st, _, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, kind="smooth")
    maps = {l: edge_ramp(images[l].shape, 64) for l in labels}
    st.camera_weights, st.blend_bands = maps, 5
    got = st.stitch(images)
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    ref = multiband_model.blend_cv2(flat.layers, flat.out_w, flat.out_h, [images[l] for l in labels],
                                    [maps[l] for l in labels], 5)
    assert np.array_equal(got, ref), _diff(got, ref)
    COVERED["cv2_full"] += 1


def test_the_file_reached_what_it_claims():
    assert len(COVERED["rigs"]) >= 20, COVERED["rigs"]
    assert COVERED["bands"] == set(range(1, 7)), COVERED["bands"]
    assert COVERED["channels"] == {1, 3, 4}
    assert COVERED["frames"] == {1, 15, 16, 17, 33, 64}
    assert COVERED["most_over_4"] == 3 and COVERED["sequence"] == 1 and COVERED["cv2_full"] == 1
    assert len(COVERED["layouts"]) == 4
