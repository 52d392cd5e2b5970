"""Shared builders of the camera-weight tests: chains, weight maps of every kind, and the layer model
evaluated on the product's own plan flattening."""
import numpy as np

from helpers import synthetic_chain
from multicamera_stitching_b200 import edge_ramp
from multicamera_stitching_b200.plan import flatten_chain
from oracle import camera_weight_model, stitcher_ref

SUPER_TRIM = (9, 5)   # super-mode crops this many pixels inside every stage canvas: several cameras stay
MAP_KINDS = ("random", "binary", "ramp", "absent", "mixed", "tiny", "rim")   # "mixed" cycles the first four


def make_maps(images, labels, kind, seed=0):
    """``{label: uint8 map or None}`` of one kind for every camera."""
    rng = np.random.default_rng(seed)
    out = {}
    for i, l in enumerate(labels):
        h, w = images[l].shape[:2]
        k = kind if kind != "mixed" else MAP_KINDS[i % 4]
        if k == "random":
            m = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
            m[rng.random((h, w)) < 0.1] = 0
        elif k == "binary":
            m = np.full((h, w), 255, np.uint8)
            m[int(h * 0.85):] = 0                       # a chassis along the bottom of the frame
            m[:h // 5, :w // 6] = 0                     # a lens-hood corner
        elif k == "ramp":
            m = edge_ramp((h, w), 1 + (i * 7) % 24)
        elif k == "tiny":                               # weights 0..3: sampled weights of 0 and 1, small sums
            m = rng.integers(0, 4, size=(h, w), dtype=np.uint8)
        elif k == "rim":                                # 255 inside a ring of 1 and a one-pixel border of 0
            m = np.zeros((h, w), np.uint8)
            m[1:h - 1, 1:w - 1] = 1
            m[2:h - 2, 2:w - 2] = 255
        else:
            m = None
        out[l] = m
    return out


def trimmed_super_chain(n, h, w, c, trim=SUPER_TRIM, kind="noise", frame_index=0):
    """A super-mode chain whose crops trim a few pixels off every stage canvas (the synthetic default
    limits keep only the newest camera): ``(stitcher, oracle states, labels, images)``."""
    from multicamera_stitching_b200 import Stitcher, synthetic
    images = synthetic.make_frames(n, h, w, c, frame_index, kind)
    st = Stitcher(images, super_mode=True)
    labels = list(st.img_labels)
    shapeB = tuple(images[labels[0]].shape)
    states = []
    for k in range(n - 1):
        sb = st.stitchers[k]
        sb.set_homography(synthetic.make_homography(k, h, w, shapeB[1]), shapeA=images[labels[k + 1]].shape,
                          shapeB=shapeB, xoffset=0, yoffset=0)
        sb.x_limits = [trim[0], sb.ABSize[0] - trim[0]]
        sb.y_limits = [trim[1], sb.ABSize[1] - trim[1]]
        shapeB = sb.result_shape()
        ost = stitcher_ref.new_state(sid=str(k), super_mode=True)
        for f in ("cachedBH", "cachedBINVH", "Bpts", "BimgSize", "cachedAH", "cachedAINVH", "Apts", "AimgSize",
                  "ABSize", "x_limits", "y_limits"):
            ost[f] = getattr(sb, f)
        states.append(ost)
    return st, states, labels, images


def chain_case(n, h, w, c, super_mode=False, frame_index=0):
    if super_mode:
        return trimmed_super_chain(n, h, w, c, frame_index=frame_index)
    return synthetic_chain(n, h, w, c, kind="noise", xoffset=3, yoffset=5, frame_index=frame_index)


def layer_model(st, labels, images, maps):
    """The layer model on the product's flattening: ``(panorama, contributions per layer, most contributors)``."""
    flat = flatten_chain(st.stitchers, [images[l].shape for l in labels])
    return camera_weight_model.blend(flat.layers, flat.out_w, flat.out_h, [images[l] for l in labels],
                                     [maps.get(l) for l in labels])
