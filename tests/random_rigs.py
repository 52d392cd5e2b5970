"""Seeded random rigs: camera counts, frame sizes, channel counts, canvas offsets, super mode and
homographies well outside the benchmark's near-identity ones (rotation, anisotropic scale, perspective,
mirrored axes), as product stitchers plus the oracle's dict states."""
import math

import numpy as np

from multicamera_stitching_b200 import Stitcher
from oracle import stitcher_ref


def mirrored(seed):
    """Whether ``random_chain(seed)`` has a mirrored camera (its first stage's)."""
    return seed % 7 == 6


def random_chain(seed, trim=None):
    """``(stitcher, oracle states, labels, images)`` of seed ``seed``, or None where a stage canvas is
    degenerate or too large.  Seeds with ``seed % 4 == 3`` are super-mode chains; their crops keep only the
    newest camera unless ``trim = (tx, ty)`` is given, which sets every stage's ``x_limits`` / ``y_limits``
    that many pixels inside ``ABSize`` instead, so that the cropped canvases keep several cameras."""
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(2, 6))
    c = int(rng.choice([1, 3, 3, 4]))
    h = int(rng.integers(24, 260))
    w = int(rng.integers(2, 22)) * 16                     # 16-byte rows at every channel count: the tiled variant applies
    if seed % 5 == 4:
        w += int(rng.integers(1, 4))                      # odd rows: the gather variant serves them
    super_mode = bool(seed % 4 == 3)
    xo, yo = int(rng.integers(0, 30)), int(rng.integers(0, 30))
    shape = (h, w) if c == 1 else (h, w, c)
    images = {"CAM%d" % (k + 1): rng.integers(0, 256, size=shape, dtype=np.uint8) for k in range(n)}
    st = Stitcher(images, super_mode=super_mode)
    labels = list(st.img_labels)
    states = []
    shapeB = shape
    for k in range(n - 1):
        ang = math.radians(rng.uniform(-12, 12))
        sx, sy = rng.uniform(0.7, 1.3, size=2)
        if mirrored(seed) and k == 0:
            sx = -sx                                      # a mirrored camera
        A = np.array([[sx * math.cos(ang), -sy * math.sin(ang) + rng.uniform(-0.1, 0.1), 0.0],
                      [sx * math.sin(ang), sy * math.cos(ang), 0.0], [0.0, 0.0, 1.0]])
        A[0, 2] = shapeB[1] * rng.uniform(0.3, 0.9) + (w if sx < 0 else 0)
        A[1, 2] = rng.uniform(-0.2, 0.2) * h
        A[2, 0], A[2, 1] = rng.uniform(-2e-4, 2e-4, size=2)
        sb = st.stitchers[k]
        sb.set_homography(A, shapeA=shape, shapeB=shapeB, xoffset=xo, yoffset=yo)
        ost = stitcher_ref.new_state(sid=str(k), super_mode=super_mode)
        stitcher_ref.geometry_from_homography(ost, A, shape, shapeB, xo, yo)
        if super_mode and trim is not None:
            sb.x_limits = [trim[0], sb.ABSize[0] - trim[0]]
            sb.y_limits = [trim[1], sb.ABSize[1] - trim[1]]
            ost["x_limits"], ost["y_limits"] = list(sb.x_limits), list(sb.y_limits)
        states.append(ost)
        shapeB = sb.result_shape()
        if shapeB[0] <= 0 or shapeB[1] <= 0 or shapeB[0] * shapeB[1] > 40e6:
            return None
    return st, states, labels, images
