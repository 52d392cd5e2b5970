"""Exposure compensation on the GPU (csrc/mcs_exposure.cu and the GAIN instantiations of the per-frame kernels): every
comparison is ``np.array_equal`` against ``oracle/exposure_model.py`` on the plan's own flattening.

- the seeded random rigs with 3 channels, every camera at its own brightness scale: the device's N, I and gains equal
  ``stats`` / ``solve`` bit for bit, and the panoramas equal the model in variant 5 (where the rig takes it) and in
  variant 6 with no seams, Voronoi seams or graph-cut seams (found on the compensated samples), numpy and device frames;
- F = 1, 16, 17 and 64, SequencePipeline into a poisoned output, strided sources;
- gains set directly (exact halves, 0, above 1 with saturation) on 1, 3 and 4 channels, and switching off;
- the C ABI's error paths, each leaving the plan unchanged;
- one full-size config-2 frame-set with cameras scaled 0.7-1.3 against the cv2 chain (GainCompensator, then
  MultiBandBlender)."""
import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, chain_case, make_maps
from multicamera_stitching_b200 import _cabi, edge_ramp
from multicamera_stitching_b200.plan import flatten_chain
from oracle import exposure_model as ex
from oracle import multiband_model as mb
from random_rigs import random_chain

pytestmark = pytest.mark.gpu

COVERED = {"rigs": set(), "stats": 0, "variants": set(), "seams": set(), "frames": set(), "entry": set(),
           "strided": 0, "direct": set(), "off": 0, "errors": 0, "cv2_full": 0}


def _scaled(images, labels, seed, lo=0.7, hi=1.3):
    """Every camera's frames at its own brightness scale."""
    rng = np.random.default_rng(1000 + seed)
    return {l: np.clip(images[l].astype(np.float64) * rng.uniform(lo, hi), 0, 255).astype(np.uint8) for l in labels}


def _check_stats(handle, flat, frames, maps, cuda_device):
    """Device N, I and gains against ``stats`` / ``solve``, bit for bit.  Returns the gains by camera."""
    import torch
    dev = [torch.from_numpy(frames[l.cam]).to(cuda_device) for l in flat.layers]
    gains, N, I = handle.estimate_gains([t.data_ptr() for t in dev], [t.stride(0) for t in dev], stats=True)
    planes = mb.camera_planes(flat.layers, flat.out_w, flat.out_h, frames, maps)
    wN, wI, skip = ex.stats(*ex.plane_inputs(planes))
    assert np.array_equal(N, wN), (N, wN)
    assert np.array_equal(I, wI), np.abs(I - wI).max()
    want = ex.solve(wN, wI, skip)
    fed = handle.fed_layers()
    assert np.array_equal(gains[fed], want), (gains[fed], want)
    assert all(gains[k] == 1.0 for k in range(len(flat.layers)) if k not in fed)
    COVERED["stats"] += 1
    out = [1.0] * (max(l.cam for l in flat.layers) + 1)
    for k, l in enumerate(flat.layers):
        out[l.cam] = float(gains[k])
    return out


@pytest.mark.parametrize("seed", range(28))
def test_random_rig_matches_the_specification(cuda_device, seed):
    import torch
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    if images[labels[0]].ndim != 3 or images[labels[0]].shape[2] != 3:
        pytest.skip("GainCompensator estimates on 3 channels")
    images = _scaled(images, labels, seed)
    maps = make_maps(images, labels, MAP_KINDS[seed % 7], seed=seed)
    frames, m = [images[l] for l in labels], [maps.get(l) for l in labels]
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    st.camera_weights = maps
    # variant 5, where the camera-weighted kernel takes the rig
    try:
        plan = st.plan([images[l].shape for l in labels], cuda_device)
    except _cabi.McsError as e:
        assert e.code == _cabi.MCS_ERR_UNSUPPORTED
        plan = None
    if plan is not None:
        gains = _check_stats(plan.handle, flat, frames, m, cuda_device)
        got = st.compensate_exposure(images)
        assert [got[str(l)] for l in labels] == [gains[c] for c in range(len(labels))]
        ref = ex.blend_weighted(flat.layers, flat.out_w, flat.out_h, frames, m, gains)
        assert np.array_equal(st.stitch(images), ref)
        assert st.plan([images[l].shape for l in labels], cuda_device).handle.last_variant() == 5
        COVERED["variants"].add(5)
    # variant 6, with no seams, Voronoi or graph-cut seams
    bands = 1 + seed % 6
    seams = (None, "voronoi", "graphcut")[seed % 3]
    st.blend_bands, st.voronoi_seams = bands, seams == "voronoi"
    gains = [float(v) for v in st.compensate_exposure(images).values()]
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    assert plan.handle.exposure_gains is not None
    if seams == "graphcut":
        st.find_graphcut_seams(images)
        plan = st.plan([images[l].shape for l in labels], cuda_device)
        assert plan.handle.graphcut_seams
    assert gains == _check_stats(plan.handle, flat, frames, m, cuda_device)[:len(labels)]
    ref = ex.blend_multiband(flat.layers, flat.out_w, flat.out_h, frames, m, bands, gains, seams=seams)
    assert np.array_equal(st.stitch(images), ref), (bands, seams)
    dev = st.stitch({l: torch.from_numpy(images[l]).to(cuda_device) for l in labels}).cpu().numpy()
    assert np.array_equal(dev, ref)
    assert plan.handle.last_variant() == 6
    COVERED["variants"].add(6)
    COVERED["seams"].add(seams)
    COVERED["rigs"].add(seed)


@pytest.mark.parametrize("F", [1, 16, 17, 64])
def test_frame_counts_and_entry_points(cuda_device, F):
    import torch
    st, states, labels, images = chain_case(3, 48, 80, 3)
    maps = make_maps(images, labels, "mixed", seed=F)
    m = [maps.get(l) for l in labels]
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    sets = [_scaled(chain_case(3, 48, 80, 3, frame_index=f)[3], labels, 7) for f in range(F)]
    st.camera_weights = maps
    gains = list(st.compensate_exposure(_scaled(images, labels, 7)).values())
    for bands in (0, 4):
        st.blend_bands = bands

        def ref(s):
            args = (flat.layers, flat.out_w, flat.out_h, [s[l] for l in labels], m)
            return ex.blend_multiband(*args, bands, gains) if bands else ex.blend_weighted(*args, gains)

        batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
        out = st.stitch_batch(batch).cpu().numpy()
        for f in range(F):
            assert np.array_equal(out[f], ref(sets[f])), (bands, f)
        plan = st.plan([images[l].shape for l in labels], cuda_device)
        assert plan.handle.last_variant() == (6 if bands else 5)
        last = sets[-1]
        got = plan.run({k: torch.from_numpy(last[l]).to(cuda_device) for k, l in enumerate(labels)}).cpu().numpy()
        assert np.array_equal(got, ref(last))
        assert np.array_equal(st.stitch(last), ref(last))
    COVERED["entry"].update(("stitch_batch", "plan", "stitch"))
    COVERED["frames"].add(F)


def test_sequence_pipeline_into_a_poisoned_output(cuda_device):
    import torch
    from multicamera_stitching_b200.sequence import SequencePipeline
    st, states, labels, images = chain_case(4, 90, 160, 3)
    st.camera_weights = {l: edge_ramp(images[l].shape, 24) for l in labels}
    st.blend_bands = 5
    st.exposure_gains = {labels[0]: 1.25, labels[1]: 0.5, labels[2]: 0.0, labels[3]: 2.5}
    F = 7
    sets = [chain_case(4, 90, 160, 3, frame_index=f)[3] for f in range(F)]
    pipe = SequencePipeline(st, [images[l].shape for l in labels], cuda_device, chunk=3, depth=2)
    assert pipe.plan.handle.exposure_gains is not None
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    m = [st.camera_weights[l] for l in labels]
    gains = [1.25, 0.5, 0.0, 2.5]

    def ref(s):
        return ex.blend_multiband(flat.layers, flat.out_w, flat.out_h, [s[l] for l in labels], m, 5, gains)

    host = {l: torch.from_numpy(np.stack([s[l] for s in sets])).pin_memory() for l in labels}
    out = torch.full((F,) + ref(images).shape, 0xEE, dtype=torch.uint8).pin_memory()
    assert pipe.run(host, out) == F
    for f in range(F):
        assert np.array_equal(out[f].numpy(), ref(sets[f])), f
    COVERED["entry"].add("SequencePipeline")


def _plan(cuda_device, c=3, n=3):
    from multicamera_stitching_b200.engine import CompiledPlan
    st, states, labels, images = chain_case(n, 60, 96, c)
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    return CompiledPlan(flat, cuda_device), flat, [images[l] for l in labels]


def test_strided_sources(cuda_device):
    """Frames that are views into wider, offset buffers, for the estimate and both blends."""
    import torch
    plan, flat, frames = _plan(cuda_device, n=4)
    h = plan.handle
    frames = [np.clip(f * s, 0, 255).astype(np.uint8) for f, s in zip(frames, (0.8, 1.2, 1.0, 0.9))]
    maps = [edge_ramp(f.shape, 12) for f in frames]
    h.set_camera_weights(maps)

    def strided(f):
        hh, ww, c = f.shape
        big = torch.zeros((hh + 3, ww + 13, c), dtype=torch.uint8, device=cuda_device)
        big[2:2 + hh, 5:5 + ww] = torch.from_numpy(f).to(cuda_device)
        return big[2:2 + hh, 5:5 + ww]

    dev = [strided(f) for f in frames]
    gains = h.estimate_gains([t.data_ptr() for t in dev], [t.stride(0) for t in dev])
    by_cam = _check_stats(h, flat, frames, maps, cuda_device)
    assert np.array_equal(gains, [by_cam[l.cam] for l in flat.layers])
    h.set_exposure_gains(gains)
    args = (flat.layers, flat.out_w, flat.out_h, frames, maps)
    assert np.array_equal(plan.run(dev).cpu().numpy(), ex.blend_weighted(*args, by_cam))
    h.set_multiband(3)
    assert np.array_equal(plan.run(dev).cpu().numpy(), ex.blend_multiband(*args, 3, by_cam))
    COVERED["strided"] += 1


@pytest.mark.parametrize("c", [1, 3, 4])
def test_gains_set_directly_and_switched_off(cuda_device, c):
    import torch
    plan, flat, frames = _plan(cuda_device, c=c)
    h = plan.handle
    dev = [torch.from_numpy(f).to(cuda_device) for f in frames]
    maps = [None] * len(frames)
    args = (flat.layers, flat.out_w, flat.out_h, frames, maps)
    h.set_camera_weights(maps)
    plain = plan.run(dev).cpu().numpy()
    for gains in ([0.5, 1.5, 2.5], [0.0, 1.0, 3.75], [1.0, 1.0, 1.0]):
        h.set_exposure_gains(gains)
        got = plan.run(dev).cpu().numpy()
        assert np.array_equal(got, ex.blend_weighted(*args, gains)), gains
        if gains[0] == 0.0:
            assert got.max() == 255   # a saturating gain
        assert np.array_equal(got, plain) == (gains == [1.0, 1.0, 1.0])
    h.set_exposure_gains(None)
    assert np.array_equal(plan.run(dev).cpu().numpy(), plain)
    h.set_multiband(4)
    plain = plan.run(dev).cpu().numpy()
    h.set_exposure_gains([2.5, 0.5, 1.5])
    assert np.array_equal(plan.run(dev).cpu().numpy(), ex.blend_multiband(*args, 4, [2.5, 0.5, 1.5]))
    h.set_exposure_gains(None)
    assert np.array_equal(plan.run(dev).cpu().numpy(), plain)
    COVERED["direct"].add(c)
    COVERED["off"] += 1


def test_error_paths_of_the_c_abi(cuda_device):
    import torch
    plan, flat, frames = _plan(cuda_device)
    h = plan.handle
    dev = [torch.from_numpy(f).to(cuda_device) for f in frames]
    ptrs, pitch = [t.data_ptr() for t in dev], [t.stride(0) for t in dev]
    with pytest.raises(_cabi.McsError, match="code -1"):   # no camera weights
        h.set_exposure_gains([1.0, 1.0, 1.0])
    with pytest.raises(_cabi.McsError, match="code -1"):
        h.estimate_gains(ptrs, pitch)
    h.set_camera_weights([None] * 3)
    h.set_exposure_gains([1.5, 0.5, 1.0])
    want = ex.blend_weighted(flat.layers, flat.out_w, flat.out_h, frames, [None] * 3, [1.5, 0.5, 1.0])
    assert np.array_equal(plan.run(dev).cpu().numpy(), want)
    for bad in ([1.0, -0.5, 1.0], [1.0, float("nan"), 1.0], [float("inf"), 1.0, 1.0]):
        with pytest.raises(_cabi.McsError, match="code -1"):
            h.set_exposure_gains(bad)
        assert np.array_equal(plan.run(dev).cpu().numpy(), want)
    # set_camera_weights clears the gains, and so does clearing the weights
    h.set_camera_weights([None] * 3)
    assert h.exposure_gains is None
    plain = ex.blend_weighted(flat.layers, flat.out_w, flat.out_h, frames, [None] * 3, [1.0] * 3)
    assert np.array_equal(plan.run(dev).cpu().numpy(), plain)
    h.set_exposure_gains([1.5, 0.5, 1.0])
    h.set_camera_weights(None)
    h.set_camera_weights([None] * 3)
    assert np.array_equal(plan.run(dev).cpu().numpy(), plain)
    # estimating on 1 or 4 channels: refused, the plan unchanged
    for c in (1, 4):
        p4, f4, fr4 = _plan(cuda_device, c=c)
        p4.handle.set_camera_weights([None] * 3)
        p4.handle.set_exposure_gains([0.5, 1.0, 1.5])
        d4 = [torch.from_numpy(f).to(cuda_device) for f in fr4]
        before = p4.run(d4).cpu().numpy()
        with pytest.raises(_cabi.McsError, match="code -3"):
            p4.handle.estimate_gains([t.data_ptr() for t in d4], [t.stride(0) for t in d4])
        assert np.array_equal(p4.run(d4).cpu().numpy(), before)
    COVERED["errors"] += 1


def test_full_size_config2_against_cv2(cuda_device):
    from multicamera_stitching_b200 import synthetic
    n, h, w = synthetic.CONFIGS["cfg2_6x1080p"]
    st, _, labels, images = synthetic.synthetic_stitcher(n, h, w, 3, kind="smooth")
    images = _scaled(images, labels, 2)
    maps = {l: edge_ramp(images[l].shape, 64) for l in labels}
    st.camera_weights, st.blend_bands = maps, 5
    got_gains = st.compensate_exposure(images)
    plan = st.plan([images[l].shape for l in labels])
    flat = plan.flat
    frames, m = [images[l] for l in labels], [maps[l] for l in labels]
    want = ex.camera_gains(flat.layers, flat.out_w, flat.out_h, frames, m, ex.gains_cv2)
    for l, g, wg in zip(labels, [got_gains[str(l)] for l in labels], want):
        assert abs(g - wg) <= 1e-12 * abs(wg) and np.array_equal(ex.lut(g), ex.lut(wg)), (l, g, wg)
    assert max(want) / min(want) > 1.2
    got = st.stitch(images)
    ref = ex.blend_multiband_cv2(flat.layers, flat.out_w, flat.out_h, frames, m, 5)
    assert np.array_equal(got, ref), int(np.abs(got.astype(int) - ref.astype(int)).max())
    COVERED["cv2_full"] += 1


def test_the_file_reached_what_it_claims():
    assert len(COVERED["rigs"]) >= 8, COVERED["rigs"]
    assert COVERED["stats"] >= 20, COVERED["stats"]
    assert COVERED["variants"] == {5, 6} and COVERED["seams"] == {None, "voronoi", "graphcut"}
    assert COVERED["frames"] == {1, 16, 17, 64}
    assert COVERED["entry"] == {"stitch", "stitch_batch", "plan", "SequencePipeline"}
    assert COVERED["strided"] == 1 and COVERED["direct"] == {1, 3, 4} and COVERED["off"] == 3
    assert COVERED["errors"] == 1 and COVERED["cv2_full"] == 1
