"""Shared builders for the tests: synthetic chains in both the product classes
and the oracle's dict states."""
import math

import numpy as np

from multicamera_stitching_b200 import Stitcher, synthetic
from oracle import stitcher_ref


def synthetic_chain(n_cams, h, w, channels=3, super_mode=False, kind="smooth", frame_index=0,
                    xoffset=0, yoffset=0, use_points_first=False):
    """Returns (stitcher, oracle_states, labels, images_dic): the product's synthetic stitcher plus the
    oracle's dict states calibrated from the same stage homographies."""
    st, homographies, labels, images = synthetic.synthetic_stitcher(
        n_cams, h, w, channels, super_mode=super_mode, kind=kind, frame_index=frame_index, xoffset=xoffset,
        yoffset=yoffset, use_points_first=use_points_first)
    states = stitcher_ref.calibrate_chain_from_homographies([images[l].shape for l in labels], homographies,
                                                            super_mode=super_mode, xoffset=xoffset, yoffset=yoffset)
    for k, ost in enumerate(states):
        ost["sid"] = str(k)
    return st, states, labels, images


def compare_u8(got, ref):
    """(max abs diff, fraction exactly equal)."""
    got = np.asarray(got)
    ref = np.asarray(ref)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    d = np.abs(got.astype(np.int16) - ref.astype(np.int16))
    return int(d.max()) if d.size else 0, float((d == 0).mean()) if d.size else 1.0


# (batch, nq_max, queries per CTA) - one geometry per path of the Hamming launcher (csrc/mcs_match.cu), which
# steps qpc down from 32 while ceil(nq_max / qpc) * batch < 2 * 148; pinned by oracle.match_model.match_qpc
MATCH_QPC_GEOMETRIES = [(1, 2000, 8), (3, 2000, 16), (4, 2000, 24), (4, 2400, 32)]


def sum_of_squares_desc(total, dim=128):
    """An integer-valued float32 descriptor in 0..255 whose squared norm is ``total`` (greedy, largest part first)."""
    d = np.zeros(dim, np.float32)
    for k in range(dim):
        v = min(255, math.isqrt(total))
        d[k], total = v, total - v * v
    assert total == 0
    return d
