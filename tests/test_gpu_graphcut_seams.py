"""Graph-cut seams of the multi-band blend on the GPU (csrc/mcs_seams_graphcut.cu): every comparison is
``np.array_equal`` against ``oracle/graphcut_seam_model.find_graphcut`` (the cut weights, read back per layer) and
``oracle/graphcut_seam_model.blend_graphcut`` (the panorama) on the plan's own flattening.

- the seeded random rigs with 3 channels on textured content, and each also on flat content, identical content
  (every camera the same frame) or masks with zero holes and borders - flat and identical content have many
  minimum cuts, where only the minimal source side makes the answer unique;
- frame counts around the 16-frame workspace sub-batch, every entry point, and SequencePipeline into a poisoned
  output;
- cases on which the terminal cost, the penalty and the 10-pixel gap each decide pixels;
- the C ABI's error paths, switching Voronoi <-> graph cut <-> none, and re-finding on a new frame-set;
- one full-height two-camera rig against the restatement and cv2's GraphCutSeamFinder directly (they differ on 4
  equal-cost pixels), the device under a time limit."""
import time

import numpy as np
import pytest

from camera_weight_cases import MAP_KINDS, SUPER_TRIM, chain_case, make_maps
from multicamera_stitching_b200 import _cabi, edge_ramp
from multicamera_stitching_b200.plan import flatten_chain
from oracle import graphcut_seam_model, multiband_model, seam_model
from random_rigs import random_chain

pytestmark = pytest.mark.gpu

COVERED = {"rigs": set(), "contents": set(), "bands": set(), "frames": set(), "layers": 0, "entry": set(),
           "sequence": 0, "cv2_full": 0, "errors": 0, "switch": 0, "refind": 0, "constants": set()}


def _flat(st, labels, images):
    return flatten_chain(st.stitchers, [images[l].shape for l in labels])


def _expected_seams(flat, seam_frames, maps, finder=graphcut_seam_model.find_graphcut):
    """``{layer index: cut weights}`` of the layers that feed the blend."""
    fed = []
    for k, l in enumerate(flat.layers):
        x0, y0, x1, y1 = [int(v) for v in l.rect]
        if min(flat.out_w, x1) > max(0, x0) and min(flat.out_h, y1) > max(0, y0):
            fed.append(k)
    planes = multiband_model.camera_planes(flat.layers, flat.out_w, flat.out_h, seam_frames, maps)
    assert len(planes) == len(fed)
    return dict(zip(fed, finder(*graphcut_seam_model.plane_inputs(planes))))


def _check_seams(handle, flat, seam_frames, maps, finder=graphcut_seam_model.find_graphcut):
    want = _expected_seams(flat, seam_frames, maps, finder)
    for k in range(len(flat.layers)):
        if k in want:
            got = handle.seam_weights(k)
            assert got.shape == want[k].shape and np.array_equal(got, want[k]), (k, int((got != want[k]).sum()))
            COVERED["layers"] += 1
        else:
            with pytest.raises(_cabi.McsError, match="code -1"):
                handle.seam_weights(k)
    return want


def _holes(images, labels, seed):
    """Masks with scattered zero pixels, zero blocks and a zero border: the 1000 penalty and zero terminals."""
    rng = np.random.default_rng(seed)
    out = {}
    for l in labels:
        h, w = images[l].shape[:2]
        m = rng.integers(1, 256, size=(h, w)).astype(np.uint8)
        m[rng.random((h, w)) < 0.04] = 0
        y, x = int(rng.integers(0, h)), int(rng.integers(0, w))
        m[y:y + h // 5, x:x + w // 5] = 0
        m[:2, :] = 0
        m[:, -3:] = 0
        out[l] = m
    return out


def _content(kind, images, labels, seed):
    """The frame-set the seams are found on."""
    if kind == "flat":
        return {l: np.full_like(images[l], 90 + seed) for l in labels}
    if kind == "identical":
        return {l: images[labels[0]].copy() for l in labels}
    return images


def _copy_pair(sizes, corners, frames, masks):
    """A plan of two pasted cameras: its planes are the frames and masks themselves."""
    from multicamera_stitching_b200.plan import LAYER_COPY, FlatPlan, Layer
    layers = [Layer(k, LAYER_COPY, None, x, y, (x, y, x + w, y + h), (h, w))
              for k, ((w, h), (x, y)) in enumerate(zip(sizes, corners))]
    out_w = max(x + w for (w, h), (x, y) in zip(sizes, corners))
    out_h = max(y + h for (w, h), (x, y) in zip(sizes, corners))
    return FlatPlan(layers, out_w, out_h, 3, 3), frames, masks


def _terminal_and_gap_case():
    """Camera 0's only own pixels are one column exactly 10 pixels left of the overlap (20 source terminals,
    200 000); the overlap costs 120 000 an edge but for one column of edges costing 8 998 (D = 4 500 and 4 497), and
    the ring above and below it 1 001 an edge: that cut costs 20 x 8 998 + 20 x 1 001 = 199 980.  At a terminal cost of
    9 999 the two tie and the minimal source side moves the cut; with a gap of 9 the source column is outside the
    submask."""
    f0 = np.full((20, 40, 3), 200, np.uint8)
    f1 = np.full((20, 40, 3), 200, np.uint8)
    f1[:, :20] = 0
    f1[:, 8] = (140, 170, 200)
    f1[:, 9] = (136, 180, 199)
    m0 = np.zeros((20, 40), np.uint8)
    m0[:, 10] = 255
    m0[:, 20:] = 255
    return _copy_pair([(40, 20), (40, 20)], [(0, 0), (20, 0)], [f0, f1], [m0, np.full((20, 40), 255, np.uint8)])


def _penalty_case(seed=281):
    """A seeded pair with zero holes in both masks whose cut moves when the penalty is 999 (found by search)."""
    rng = np.random.default_rng(seed)
    w, h = int(rng.integers(24, 40)), int(rng.integers(14, 24))
    dx = int(rng.integers(8, w - 6))
    base = rng.integers(60, 200, (h, w + dx, 3))
    amp = int(rng.integers(8, 40))
    frames = [np.clip(base[:, x:x + w] + rng.integers(-amp, amp + 1, (h, w, 3)), 0, 255).astype(np.uint8)
              for x in (0, dx)]
    masks = []
    for _ in range(2):
        m = np.full((h, w), 255, np.uint8)
        m[rng.random((h, w)) < float(rng.uniform(0.0, 0.3))] = 0
        masks.append(m)
    return _copy_pair([(w, h), (w, h)], [(0, 0), (dx, 0)], frames, masks)


@pytest.mark.parametrize("case,moved", [("terminal_and_gap", ("TERMINAL", 9999)), ("terminal_and_gap", ("GAP", 9)),
                                        ("penalty", ("PENALTY", 999))])
def test_the_constants_are_observable(cuda_device, monkeypatch, case, moved):
    """Cases on which the terminal cost, the penalty and the gap each decide pixels: moved by one in the
    restatement, the cut changes; the device equals the restatement."""
    import torch
    from multicamera_stitching_b200.engine import CompiledPlan
    flat, frames, masks = _terminal_and_gap_case() if case == "terminal_and_gap" else _penalty_case()
    want = _expected_seams(flat, frames, masks)
    with monkeypatch.context() as mp:
        mp.setattr(graphcut_seam_model, moved[0], moved[1])
        other = _expected_seams(flat, frames, masks)
    assert any(not np.array_equal(want[k], other[k]) for k in want)
    plan = CompiledPlan(flat, cuda_device, camera_weights=masks, blend_bands=3, graphcut_frames=frames)
    _check_seams(plan.handle, flat, frames, masks)
    got = plan.run([torch.from_numpy(f).to(cuda_device) for f in frames]).cpu().numpy()
    assert np.array_equal(got, graphcut_seam_model.blend_graphcut(flat.layers, flat.out_w, flat.out_h, frames, masks, 3))
    COVERED["constants"].add(moved[0])


@pytest.mark.parametrize("seed", range(28))
def test_random_rig_matches_the_specification(cuda_device, seed):
    import torch
    made = random_chain(seed, trim=SUPER_TRIM)
    if made is None:
        pytest.skip("degenerate canvas for this seed")
    st, states, labels, images = made
    if images[labels[0]].ndim != 3 or images[labels[0]].shape[2] != 3:
        pytest.skip("the colour cost takes 3 channels")
    second = ("flat", "identical", "holes")[seed % 3]
    for i, content in enumerate(("textured", second)):
        bands = 1 + (seed + i) % 6
        maps = _holes(images, labels, seed) if content == "holes" else make_maps(images, labels, MAP_KINDS[seed % 7],
                                                                                 seed=seed)
        seam = _content(content, images, labels, seed)
        st.camera_weights, st.blend_bands = maps, bands
        st.find_graphcut_seams(seam)
        plan = st.plan([images[l].shape for l in labels], cuda_device)
        assert plan.handle.graphcut_seams and not plan.handle.voronoi_seams
        flat = plan.flat
        frames, m = [images[l] for l in labels], [maps.get(l) for l in labels]
        _check_seams(plan.handle, flat, [seam[l] for l in labels], m)
        ref = graphcut_seam_model.blend_graphcut(flat.layers, flat.out_w, flat.out_h, frames, m, bands,
                                        seam_frames=[seam[l] for l in labels])
        got = st.stitch(images)
        assert got.shape == ref.shape and np.array_equal(got, ref), (content, bands)
        dev = st.stitch({l: torch.from_numpy(images[l]).to(cuda_device) for l in labels}).cpu().numpy()
        assert np.array_equal(dev, ref), (content, bands)
        assert plan.handle.last_variant() == 6
        COVERED["contents"].add(content)
        COVERED["bands"].add(bands)
    COVERED["rigs"].add(seed)


@pytest.mark.parametrize("F", [1, 16, 17])
def test_frame_counts_and_entry_points(cuda_device, F):
    import torch
    st, states, labels, images = chain_case(3, 48, 80, 3)
    maps = make_maps(images, labels, "mixed", seed=F)
    st.camera_weights, st.blend_bands = maps, 4
    st.find_graphcut_seams(images)
    m = [maps.get(l) for l in labels]
    flat = _flat(st, labels, images)
    sets = [chain_case(3, 48, 80, 3, frame_index=f)[3] for f in range(F)]

    def ref(s):
        return graphcut_seam_model.blend_graphcut(flat.layers, flat.out_w, flat.out_h, [s[l] for l in labels], m, 4,
                                         seam_frames=[images[l] for l in labels])

    batch = {l: torch.from_numpy(np.stack([s[l] for s in sets])).to(cuda_device) for l in labels}
    out = st.stitch_batch(batch).cpu().numpy()
    for f in range(F):
        assert np.array_equal(out[f], ref(sets[f])), f
    COVERED["entry"].add("stitch_batch")
    plan = st.plan([images[l].shape for l in labels], cuda_device)
    last = sets[-1]
    got = plan.run({k: torch.from_numpy(last[l]).to(cuda_device) for k, l in enumerate(labels)}).cpu().numpy()
    assert np.array_equal(got, ref(last))
    assert np.array_equal(st.stitch(last), ref(last))
    COVERED["entry"].update(("plan", "stitch"))
    COVERED["frames"].add(F)


def test_sequence_pipeline_into_a_poisoned_output(cuda_device):
    import torch
    from multicamera_stitching_b200.sequence import SequencePipeline
    st, states, labels, images = chain_case(4, 90, 160, 3)
    st.camera_weights = {l: edge_ramp(images[l].shape, 24) for l in labels}
    st.blend_bands = 5
    seam = chain_case(4, 90, 160, 3, frame_index=9)[3]
    st.find_graphcut_seams(seam)
    F = 7
    sets = [chain_case(4, 90, 160, 3, frame_index=f)[3] for f in range(F)]
    pipe = SequencePipeline(st, [images[l].shape for l in labels], cuda_device, chunk=3, depth=2)
    assert pipe.plan.handle.graphcut_seams
    flat = _flat(st, labels, images)
    m = [st.camera_weights[l] for l in labels]

    def ref(s):
        return graphcut_seam_model.blend_graphcut(flat.layers, flat.out_w, flat.out_h, [s[l] for l in labels], m, 5,
                                         seam_frames=[seam[l] for l in labels])

    host = {l: torch.from_numpy(np.stack([s[l] for s in sets])).pin_memory() for l in labels}
    out = torch.full((F,) + ref(images).shape, 0xEE, dtype=torch.uint8).pin_memory()
    assert pipe.run(host, out) == F
    for f in range(F):
        assert np.array_equal(out[f].numpy(), ref(sets[f])), f
    COVERED["sequence"] += 1
    COVERED["entry"].add("SequencePipeline")


def _plan(cuda_device, c=3, n=3):
    from multicamera_stitching_b200.engine import CompiledPlan
    st, states, labels, images = chain_case(n, 60, 96, c)
    flat = _flat(st, labels, images)
    return CompiledPlan(flat, cuda_device), flat, [images[l] for l in labels]


def _set(handle, flat, frames, cuda_device):
    import torch
    dev = [torch.from_numpy(frames[l.cam]).to(cuda_device) for l in flat.layers]
    handle.set_graphcut_seams([t.data_ptr() for t in dev], [t.stride(0) for t in dev])


def test_error_paths_of_the_c_abi(cuda_device):
    import torch
    plan, flat, frames = _plan(cuda_device)
    h = plan.handle
    dev = [torch.from_numpy(f).to(cuda_device) for f in frames]
    args = (flat.layers, flat.out_w, flat.out_h, frames, [None] * len(frames), 3)
    with pytest.raises(_cabi.McsError, match="code -1"):   # no multi-band blend
        _set(h, flat, frames, cuda_device)
    h.set_camera_weights([None] * len(flat.layers))
    with pytest.raises(_cabi.McsError, match="code -1"):   # the single-band blend takes no seams
        _set(h, flat, frames, cuda_device)
    h.set_multiband(3)
    with pytest.raises(_cabi.McsError, match="code -1"):
        h.seam_weights(0)
    _set(h, flat, frames, cuda_device)
    assert h.graphcut_seams
    _check_seams(h, flat, frames, [None] * len(frames))
    cut = graphcut_seam_model.blend_graphcut(*args)
    assert np.array_equal(plan.run(dev).cpu().numpy(), cut)
    # set_multiband switches the seams off
    h.set_multiband(3)
    assert not h.graphcut_seams
    with pytest.raises(_cabi.McsError, match="code -1"):
        h.seam_weights(0)
    assert np.array_equal(plan.run(dev).cpu().numpy(), multiband_model.blend(*args))
    # so does set_camera_weights, and the multi-band blend with them
    _set(h, flat, frames, cuda_device)
    h.set_camera_weights([None] * len(flat.layers))
    assert not h.graphcut_seams and not h.multiband
    with pytest.raises(_cabi.McsError, match="code -1"):
        _set(h, flat, frames, cuda_device)
    # 1 and 4 channels: refused, the plan unchanged
    for c in (1, 4):
        p4, f4, fr4 = _plan(cuda_device, c=c)
        p4.handle.set_camera_weights([None] * len(f4.layers))
        p4.handle.set_multiband(3)
        d4 = [torch.from_numpy(f).to(cuda_device) for f in fr4]
        before = p4.run(d4).cpu().numpy()
        with pytest.raises(_cabi.McsError, match="code -3"):
            p4.handle.set_graphcut_seams([t.data_ptr() for t in d4], [t.stride(0) for t in d4])
        assert not p4.handle.graphcut_seams and p4.handle.multiband
        assert np.array_equal(p4.run(d4).cpu().numpy(), before)
    COVERED["errors"] += 1


def test_switching_voronoi_graphcut_and_none(cuda_device):
    import torch
    plan, flat, frames = _plan(cuda_device, n=4)
    h = plan.handle
    maps = [edge_ramp(f.shape, 9) for f in frames]
    h.set_camera_weights(maps)
    h.set_multiband(4)
    dev = [torch.from_numpy(f).to(cuda_device) for f in frames]
    args = (flat.layers, flat.out_w, flat.out_h, frames, maps, 4)
    none, voronoi, graphcut = multiband_model.blend(*args), seam_model.blend(*args), graphcut_seam_model.blend_graphcut(*args)
    assert not np.array_equal(voronoi, graphcut) and not np.array_equal(none, graphcut)
    for step in ("graphcut", "voronoi", "graphcut", "none", "graphcut", "graphcut", "voronoi-off"):
        if step == "graphcut":
            _set(h, flat, frames, cuda_device)
            assert h.graphcut_seams and not h.voronoi_seams
            want = graphcut
        elif step == "voronoi":
            h.set_voronoi_seams(True)
            assert h.voronoi_seams and not h.graphcut_seams
            want = voronoi
        elif step == "none":
            h.set_graphcut_seams(None, None)
            assert not h.graphcut_seams and h.blend_bands == 4
            with pytest.raises(_cabi.McsError, match="code -1"):
                h.seam_weights(0)
            want = none
        else:
            h.set_voronoi_seams(False)   # switches graph-cut seams off too
            assert not h.graphcut_seams and not h.voronoi_seams
            want = none
        assert np.array_equal(plan.run(dev).cpu().numpy(), want), step
    h.set_graphcut_seams(None, None)    # off twice
    assert np.array_equal(plan.run(dev).cpu().numpy(), none)
    COVERED["switch"] += 1


def test_a_new_frame_set_finds_new_seams(cuda_device):
    st, states, labels, images = chain_case(3, 64, 112, 3)
    st.blend_bands = 3
    other = chain_case(3, 64, 112, 3, frame_index=5)[3]
    st.find_graphcut_seams(images)
    first = st.plan([images[l].shape for l in labels], cuda_device)
    masks_a = [first.handle.seam_weights(k) for k in range(len(first.flat.layers))]
    out_a = st.stitch(images)
    st.find_graphcut_seams(other)
    second = st.plan([images[l].shape for l in labels], cuda_device)
    assert second is not first
    masks_b = [second.handle.seam_weights(k) for k in range(len(second.flat.layers))]
    assert any(not np.array_equal(a, b) for a, b in zip(masks_a, masks_b))
    flat = second.flat
    m = [None] * len(labels)
    _check_seams(second.handle, flat, [other[l] for l in labels], m)
    ref = graphcut_seam_model.blend_graphcut(flat.layers, flat.out_w, flat.out_h, [images[l] for l in labels], m, 3,
                                    seam_frames=[other[l] for l in labels])
    out_b = st.stitch(images)
    assert np.array_equal(out_b, ref) and not np.array_equal(out_a, out_b)
    st.find_graphcut_seams(images)   # the first frame-set again: the first plan, from the cache
    assert st.plan([images[l].shape for l in labels], cuda_device) is first
    COVERED["refind"] += 1


def test_full_height_rig_against_cv2(cuda_device):
    from multicamera_stitching_b200 import synthetic
    from multicamera_stitching_b200.engine import CompiledPlan
    st, _, labels, images = synthetic.synthetic_stitcher(2, 1080, 640, 3, kind="smooth")
    flat = _flat(st, labels, images)
    frames = [images[l] for l in labels]
    maps = [edge_ramp(f.shape, 64) for f in frames]
    t0 = time.perf_counter()
    plan = CompiledPlan(flat, cuda_device, camera_weights=maps, blend_bands=5, graphcut_frames=frames)
    elapsed = time.perf_counter() - t0
    assert plan.handle.graphcut_seams
    assert elapsed < 20.0, elapsed
    want = _check_seams(plan.handle, flat, frames, maps)   # the restatement, bit for bit (scipy: ~30 s)
    assert sum(int(v.size) for v in want.values()) > 1_000_000
    # cv2 directly: the same cut but for equal-cost ties, 4 pixels of this rig where the restatement differs from cv2
    # in the same way (its search order picks another minimum cut)
    ref = _expected_seams(flat, frames, maps, graphcut_seam_model.find_graphcut_cv2)
    differ = sum(int((want[k] != ref[k]).sum()) for k in want)
    assert differ <= 16, differ
    COVERED["cv2_full"] += 1


def test_the_file_reached_what_it_claims():
    assert len(COVERED["rigs"]) >= 8, COVERED["rigs"]
    assert COVERED["contents"] == {"textured", "flat", "identical", "holes"}, COVERED["contents"]
    assert COVERED["bands"] == set(range(1, 7)), COVERED["bands"]
    assert COVERED["frames"] == {1, 16, 17}
    assert COVERED["entry"] == {"stitch", "stitch_batch", "plan", "SequencePipeline"}
    assert COVERED["layers"] >= 40, COVERED["layers"]
    assert COVERED["sequence"] == 1 and COVERED["cv2_full"] == 1 and COVERED["errors"] == 1
    assert COVERED["switch"] == 1 and COVERED["refind"] == 1
    assert COVERED["constants"] == {"TERMINAL", "GAP", "PENALTY"}
