"""B200-native frame-compositing hot path of kiwicampus/multicamera_stitching.

``Stitcher`` / ``StitcherBase`` mirror the reference's
``PostScripts/Stitcher/StitcherClass.py``; the per-frame warp + paste and the
recalibration matcher / RANSAC run as hand-written sm_100a kernels behind the
C ABI declared in ``include/mcs.h`` (``libmcs_b200.so``).
"""
from .StitcherClass import Stitcher, StitcherBase, edge_ramp  # noqa: F401
from .Utils import (CalculateProjectionMatrix, get_projection_point_dst,  # noqa: F401
                    get_projection_point_src)

__all__ = ["Stitcher", "StitcherBase", "edge_ramp", "CalculateProjectionMatrix",
           "get_projection_point_dst", "get_projection_point_src"]
