"""Camera-weighted blend on the GPU: mcs_stitch_weighted_kernel equals the layer model of
oracle/camera_weight_model.py bit for bit, through every entry point that takes the mode."""
import numpy as np
import pytest

from camera_weight_cases import chain_case, layer_model, make_maps
from multicamera_stitching_b200 import _cabi, edge_ramp
from multicamera_stitching_b200.plan import LAYER_COPY, LAYER_REMAP, LAYER_WARP, FlatPlan, Layer, PlanUnsupported
from oracle import camera_weight_model, stitcher_ref

pytestmark = pytest.mark.gpu


def _ramps(images, labels, width=16):
    return {l: edge_ramp(images[l].shape, width) for l in labels}


@pytest.mark.parametrize("n,h,w,c,super_mode,kind", [
    (2, 64, 96, 3, False, "random"), (3, 90, 160, 1, False, "binary"), (4, 72, 120, 4, False, "ramp"),
    (5, 48, 80, 3, False, "absent"), (8, 40, 64, 3, False, "mixed"), (3, 120, 200, 3, True, "ramp"),
    (4, 90, 160, 4, True, "random"), (6, 48, 96, 1, True, "mixed"), (6, 270, 480, 3, False, "ramp"),
])
def test_kernel_matches_the_layer_model(cuda_device, n, h, w, c, super_mode, kind):
    st, states, labels, images = chain_case(n, h, w, c, super_mode)
    maps = make_maps(images, labels, kind, seed=n * 10 + c)
    st.camera_weights = maps
    ref, contrib, _ = layer_model(st, labels, images, maps)
    got = st.stitch(images)
    assert got.shape == ref.shape and np.array_equal(got, ref), int(np.abs(got.astype(int) - ref.astype(int)).max())
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.last_variant() == 5
    assert plan.owned_pixels() == contrib
    assert plan.algorithmic_bytes() == plan.out_w * plan.out_h * plan.channels + plan.channels * sum(contrib)
    # the mode reads whole frames
    assert all(win == (0, 0, int(l.src_hw[1]), int(l.src_hw[0]))
               for win, l in zip(plan.handle.source_windows(), plan.flat.layers))


@pytest.mark.parametrize("F", [1, 16, 17, 40])
def test_frame_loop_and_grid_z(cuda_device, F):
    import torch
    st, states, labels, images = chain_case(3, 90, 160, 3)
    maps = make_maps(images, labels, "mixed", seed=F)
    st.camera_weights = maps
    sets = [chain_case(3, 90, 160, 3, frame_index=f)[3] for f in range(F)]
    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    out = st.stitch_batch(batch).cpu().numpy()
    for f in range(F):
        assert np.array_equal(out[f], layer_model(st, labels, sets[f], maps)[0]), f


def _strided(torch, arr, pitch, offset, device):
    """``arr`` ([F,] H, W, C uint8) on the device with rows ``pitch`` bytes apart from byte ``offset`` of a buffer."""
    F, h = arr.shape[0], arr.shape[1]
    buf = torch.zeros(offset + F * h * pitch + 16, dtype=torch.uint8, device=device)
    view = torch.as_strided(buf, arr.shape, (h * pitch, pitch, arr.shape[3], 1), offset)
    view.copy_(torch.from_numpy(arr).to(device))
    return view


@pytest.mark.parametrize("w,pitch_pad,offset", [(160, 0, 0), (160, 4, 1), (131, 0, 0), (131, 3, 0), (131, 3, 2)])
def test_word_and_byte_paths_and_a_poisoned_output(cuda_device, w, pitch_pad, offset):
    import torch
    F = 5
    st, states, labels, images = chain_case(3, 80, w, 3)
    maps = make_maps(images, labels, "random", seed=w)
    st.camera_weights = maps
    sets = [chain_case(3, 80, w, 3, frame_index=f)[3] for f in range(F)]
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    frames = []
    for l in labels:
        arr = np.stack([s[l] for s in sets])
        frames.append(_strided(torch, arr, arr.shape[2] * 3 + pitch_pad, offset, cuda_device))
    row = plan.out_w * 3
    pitch = row + 29
    poison = torch.full((F, plan.out_h, pitch), 0xAB, dtype=torch.uint8, device=cuda_device)
    out = torch.as_strided(poison, (F, plan.out_h, plan.out_w, 3), (plan.out_h * pitch, pitch, 3, 1))
    plan.run(frames, out=out, n_frames=F)
    assert plan.handle.last_variant() == 5
    got = out.cpu().numpy()
    for f in range(F):
        assert np.array_equal(got[f], layer_model(st, labels, sets[f], maps)[0]), f
    assert bool((poison[:, :, row:] == 0xAB).all())


def _stack_plan(cuda_device, n_layers, h=64, w=96, c=3):
    """A rig whose cameras all see the middle of a 128 x 80 panorama: camera 0 pasted at (8, 8), the others
    warped with small shifts, shears and scales.  Returns (plan, flat, frames)."""
    from multicamera_stitching_b200 import synthetic
    from multicamera_stitching_b200.engine import CompiledPlan
    layers = [Layer(0, LAYER_COPY, None, 8, 8, (8, 8, 8 + w, 8 + h), (h, w))]
    for k in range(1, n_layers):
        H = np.array([[1 + 0.02 * k, 0.01 * k, 4 * k], [0.005 * k, 1 - 0.01 * k, 3 * k], [1e-5 * k, 0, 1]])
        layers.append(Layer(k, LAYER_WARP, H, 0, 0, (0, 0, 128, 80), (h, w)))
    flat = FlatPlan(layers, 128, 80, c, 3)
    frames = [synthetic.make_frame(h, w, c, cam_index=k, kind="noise") for k in range(n_layers)]
    return CompiledPlan(flat, cuda_device), flat, frames


def test_four_cameras_on_one_pixel_blend_and_five_are_refused(cuda_device):
    import torch
    plan, flat, frames = _stack_plan(cuda_device, 4)
    maps = [edge_ramp(f.shape, 5 + 3 * k) for k, f in enumerate(frames)]
    ref, contrib, most = camera_weight_model.blend(flat.layers, flat.out_w, flat.out_h, frames, maps)
    assert most == 4
    plan.handle.set_camera_weights(maps)
    got = plan.run([torch.from_numpy(f).to(cuda_device) for f in frames]).cpu().numpy()
    assert plan.handle.last_variant() == 5 and np.array_equal(got, ref)
    assert plan.owned_pixels() == contrib
    # the tiled kernel does not serve the mode
    plan.handle.force_variant(2)
    with pytest.raises(_cabi.McsError, match="code -3"):
        plan.run([torch.from_numpy(f).to(cuda_device) for f in frames])
    plan.handle.force_variant(0)
    # the stage-wise blend and the camera weights exclude each other
    with pytest.raises(_cabi.McsError, match="code -1"):
        plan.handle.set_feather(2)
    plan.handle.set_camera_weights(None)
    plan.handle.set_feather(2)
    with pytest.raises(_cabi.McsError, match="code -1"):
        plan.handle.set_camera_weights(maps)
    plan.handle.set_feather(0)

    plan5, flat5, frames5 = _stack_plan(cuda_device, 5)
    assert camera_weight_model.blend(flat5.layers, flat5.out_w, flat5.out_h, frames5, [None] * 5)[2] == 5
    with pytest.raises(_cabi.McsError, match="code -3"):
        plan5.handle.set_camera_weights([None] * 5)
    assert not plan5.handle.camera_weighted
    # left in the overwrite
    ts = [torch.from_numpy(f).to(cuda_device) for f in frames5]
    plan5.run(ts)
    assert plan5.handle.last_variant() in (1, 2)


def test_remap_layer(cuda_device):
    import torch
    from multicamera_stitching_b200 import prewarp, synthetic
    from multicamera_stitching_b200.engine import CompiledPlan
    W, H = 240, 120
    A = np.array([[200.0, 0, W / 2], [0, 200.0, H / 2], [0, 0, 1]])
    xy, frac = prewarp.undistort_maps(A, np.array([-0.3, 0.1, 0.001, -0.002, 0.0]), (W, H))
    layers = [Layer(0, LAYER_COPY, None, 20, 10, (20, 10, 180, 100), (90, 160)),
              Layer(1, LAYER_REMAP, None, 0, 0, (0, 0, W, H), (H, W), (xy, frac))]
    flat = FlatPlan(layers, W, H, 3, 3)
    frames = [synthetic.make_frame(90, 160, 3, cam_index=0, kind="noise"),
              synthetic.make_frame(H, W, 3, cam_index=1, kind="noise")]
    maps = [edge_ramp((90, 160), 12), make_maps({"a": frames[1]}, ["a"], "random", seed=3)["a"]]
    ref, contrib, _ = camera_weight_model.blend(layers, W, H, frames, maps)
    plan = CompiledPlan(flat, cuda_device, camera_weights=maps)
    got = plan.run([torch.from_numpy(f).to(cuda_device) for f in frames]).cpu().numpy()
    assert plan.handle.last_variant() == 5 and np.array_equal(got, ref)
    assert plan.owned_pixels() == contrib


def test_stitch_entry_points_and_sequence_pipeline(cuda_device):
    import torch
    from multicamera_stitching_b200.sequence import SequencePipeline
    st, states, labels, images = chain_case(4, 90, 160, 3)
    st.camera_weights = _ramps(images, labels)
    ref = layer_model(st, labels, images, st.camera_weights)[0]
    assert np.array_equal(st.stitch(images), ref)
    dev = {l: torch.from_numpy(images[l]).to(cuda_device) for l in labels}
    assert np.array_equal(st.stitch(dev).cpu().numpy(), ref)
    F = 6
    sets = [chain_case(4, 90, 160, 3, frame_index=f)[3] for f in range(F)]
    shapes = [images[l].shape for l in labels]
    pipe = SequencePipeline(st, shapes, cuda_device, chunk=4, depth=2)
    # whole frames go up
    assert all(len(c) == 1 and c[0]["b0"] == 0 and c[0]["nbytes"] == g[0] and c[0]["rows"] == g[1]
               for c, g in zip(pipe.windows, pipe.geometry))
    host = {l: torch.from_numpy(np.stack([s[l] for s in sets])).pin_memory() for l in labels}
    out = torch.empty((F,) + ref.shape, dtype=torch.uint8).pin_memory()
    assert pipe.run(host, out) == F
    for f in range(F):
        assert np.array_equal(out[f].numpy(), layer_model(st, labels, sets[f], st.camera_weights)[0]), f


def test_clearing_the_maps_returns_to_the_overwrite(cuda_device):
    import torch
    st, states, labels, images = chain_case(3, 90, 160, 3)
    st.camera_weights = _ramps(images, labels)
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    dev = [torch.from_numpy(images[l]).to(cuda_device) for l in labels]
    plan.run(dev)
    assert plan.handle.last_variant() == 5
    plan.handle.set_camera_weights(None)
    got = plan.run(dev).cpu().numpy()
    assert plan.handle.last_variant() == 2
    st.camera_weights = None
    fresh = st.plan([images[l].shape for l in labels], cuda_device)
    assert fresh is not plan
    assert np.array_equal(got, fresh.run(dev).cpu().numpy())
    assert np.array_equal(got, stitcher_ref.stitch_chain(states, labels, images))


def test_segmented_chains_are_refused(cuda_device):
    st, states, labels, images = chain_case(3, 90, 160, 3)
    st.camera_weights = {}
    # stage 1 calibrated for a canvas of another size: the composited canvas would be resized
    st.stitchers[1].BimgSize = (st.stitchers[1].BimgSize[0] - 2, st.stitchers[1].BimgSize[1] - 2, 3)
    with pytest.raises(PlanUnsupported, match="camera weights"):
        st.stitch(images)
