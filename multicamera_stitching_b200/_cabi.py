"""ctypes binding of ``libmcs_b200.so`` (declared in ``include/mcs.h``).

There is deliberately no fallback: if the library is missing or fails to load,
or if a call returns an error code, an exception is raised.
"""
import ctypes
import os

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# $MCS_B200_LIB points the binding at another build of the same library (comparisons between builds)
LIB_PATH = os.environ.get("MCS_B200_LIB") or os.path.join(_PKG_DIR, "libmcs_b200.so")

MCS_OK = 0
MCS_MAX_LAYERS = 16
MCS_LAYER_COPY = 0
MCS_LAYER_WARP = 1
MCS_LAYER_REMAP = 2
ABI_VERSION = 3

# every symbol include/mcs.h declares
EXPORTS = (
    "mcs_abi_version", "mcs_last_error", "mcs_plan_create", "mcs_plan_create_maps", "mcs_plan_destroy",
    "mcs_plan_owned_pixels", "mcs_plan_source_windows", "mcs_plan_source_spans", "mcs_copy_window_u8", "mcs_upload_pageable_u8", "mcs_stitch_u8", "mcs_plan_set_feather", "mcs_plan_set_blend", "mcs_plan_set_camera_weights",
    "mcs_plan_set_multiband", "mcs_plan_multiband_bands", "mcs_plan_last_variant",
    "mcs_plan_force_variant", "mcs_plan_rows_need_padding", "mcs_plan_promise_padded_rows",
    "mcs_plan_tiled_status", "mcs_plan_tiled_ctas_per_sm", "mcs_plan_tiled_stats", "mcs_launch_count",
    "mcs_match_hamming_top2", "mcs_match_l2_top2", "mcs_ransac_homography", "mcs_refit_homography", "mcs_resize_linear_u8",
)


MCS_ERR_UNSUPPORTED = -3


class McsError(RuntimeError):
    def __init__(self, msg, code=None):
        RuntimeError.__init__(self, msg)
        self.code = code


_lib = None

_c_i32p = ctypes.POINTER(ctypes.c_int32)
_c_i64p = ctypes.POINTER(ctypes.c_int64)
_c_f64p = ctypes.POINTER(ctypes.c_double)
_vp = ctypes.c_void_p


def load(build_if_missing=False):
    """Load (once) and return the ctypes handle of the library."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if build_if_missing:
            from . import build as _build
            _build.build()
        else:
            raise McsError(
                "%s not found: build it with `python -m multicamera_stitching_b200.build` "
                "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.mcs_abi_version.restype = ctypes.c_int
    lib.mcs_abi_version.argtypes = []
    if lib.mcs_abi_version() != ABI_VERSION:
        raise McsError("libmcs_b200.so ABI %d != binding ABI %d - rebuild"
                       % (lib.mcs_abi_version(), ABI_VERSION))
    lib.mcs_last_error.restype = ctypes.c_char_p
    lib.mcs_last_error.argtypes = []
    lib.mcs_plan_create.restype = ctypes.c_int
    lib.mcs_plan_create.argtypes = [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int, _c_i32p, _c_i32p,
                                    _c_f64p, _c_i32p, _c_i32p, ctypes.c_int, ctypes.c_int]
    lib.mcs_plan_create_maps.restype = ctypes.c_int
    lib.mcs_plan_create_maps.argtypes = [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int, _c_i32p, _c_i32p,
                                         _c_f64p, _c_i32p, _c_i32p, ctypes.c_int, ctypes.c_int,
                                         ctypes.POINTER(_vp), ctypes.POINTER(_vp), _c_i32p]
    lib.mcs_plan_destroy.restype = ctypes.c_int
    lib.mcs_plan_destroy.argtypes = [_vp]
    lib.mcs_plan_owned_pixels.restype = ctypes.c_int
    lib.mcs_plan_owned_pixels.argtypes = [_vp, _c_i64p, _vp]
    lib.mcs_plan_source_windows.restype = ctypes.c_int
    lib.mcs_plan_source_windows.argtypes = [_vp, _c_i32p]
    lib.mcs_plan_source_spans.restype = ctypes.c_int
    lib.mcs_plan_source_spans.argtypes = [_vp, ctypes.c_int, ctypes.c_int, _c_i32p]
    lib.mcs_copy_window_u8.restype = ctypes.c_int
    lib.mcs_copy_window_u8.argtypes = [_vp, ctypes.c_int64, ctypes.c_int64, _vp, ctypes.c_int64, ctypes.c_int64,
                                       ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]
    lib.mcs_upload_pageable_u8.restype = ctypes.c_int
    lib.mcs_upload_pageable_u8.argtypes = [ctypes.c_int, ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(_vp),
                                           _c_i64p, _c_i64p, _c_i64p, ctypes.c_int64, ctypes.c_int, _vp]
    lib.mcs_refit_homography.restype = ctypes.c_int
    lib.mcs_refit_homography.argtypes = [_vp, _vp, _vp, ctypes.c_int, _vp, ctypes.c_int, _vp]
    lib.mcs_stitch_u8.restype = ctypes.c_int
    lib.mcs_stitch_u8.argtypes = [_vp, ctypes.POINTER(_vp), _c_i64p, _c_i64p, ctypes.c_int, _vp,
                                  ctypes.c_int64, ctypes.c_int64, _vp]
    lib.mcs_plan_last_variant.restype = ctypes.c_int
    lib.mcs_plan_last_variant.argtypes = [_vp]
    lib.mcs_plan_force_variant.restype = ctypes.c_int
    lib.mcs_plan_force_variant.argtypes = [_vp, ctypes.c_int]
    lib.mcs_plan_rows_need_padding.restype = ctypes.c_int
    lib.mcs_plan_rows_need_padding.argtypes = [_vp]
    lib.mcs_plan_promise_padded_rows.restype = ctypes.c_int
    lib.mcs_plan_promise_padded_rows.argtypes = [_vp, ctypes.c_int]
    lib.mcs_plan_set_feather.restype = ctypes.c_int
    lib.mcs_plan_set_feather.argtypes = [_vp, ctypes.c_int]
    lib.mcs_plan_set_blend.restype = ctypes.c_int
    lib.mcs_plan_set_blend.argtypes = [_vp, ctypes.c_int, _c_i32p, ctypes.POINTER(ctypes.c_void_p), _c_i64p]
    lib.mcs_plan_set_camera_weights.restype = ctypes.c_int
    lib.mcs_plan_set_camera_weights.argtypes = [_vp, ctypes.POINTER(ctypes.c_void_p), _c_i64p]
    lib.mcs_plan_set_multiband.restype = ctypes.c_int
    lib.mcs_plan_set_multiband.argtypes = [_vp, ctypes.c_int]
    lib.mcs_plan_multiband_bands.restype = ctypes.c_int
    lib.mcs_plan_multiband_bands.argtypes = [_vp]
    lib.mcs_plan_tiled_ctas_per_sm.restype = ctypes.c_int
    lib.mcs_plan_tiled_ctas_per_sm.argtypes = [_vp]
    lib.mcs_plan_tiled_status.restype = ctypes.c_char_p
    lib.mcs_plan_tiled_status.argtypes = [_vp]
    lib.mcs_plan_tiled_stats.restype = ctypes.c_int
    lib.mcs_plan_tiled_stats.argtypes = [_vp, _c_i32p]
    lib.mcs_launch_count.restype = ctypes.c_int64
    lib.mcs_launch_count.argtypes = []
    lib.mcs_match_hamming_top2.restype = ctypes.c_int
    lib.mcs_match_hamming_top2.argtypes = [_vp, _vp, ctypes.c_int, _vp, _vp, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_double, _vp, _vp, _vp, ctypes.c_int, _vp]
    lib.mcs_ransac_homography.restype = ctypes.c_int
    lib.mcs_match_l2_top2.restype = ctypes.c_int
    lib.mcs_match_l2_top2.argtypes = [_vp, _vp, ctypes.c_int, _vp, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                      _vp, _vp, _vp, ctypes.c_int, _vp]
    lib.mcs_ransac_homography.argtypes = [_vp, _vp, _vp, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_float,
                                          _vp, _vp, _vp, _vp, ctypes.c_int, _vp]
    lib.mcs_resize_linear_u8.restype = ctypes.c_int
    lib.mcs_resize_linear_u8.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int64,
                                         _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int64,
                                         ctypes.c_int, ctypes.c_int, _vp]
    _lib = lib
    return lib


def check(rc, what):
    if rc != MCS_OK:
        msg = load().mcs_last_error().decode(errors="replace")
        raise McsError("%s failed (code %d): %s" % (what, rc, msg), rc)


def launch_count():
    return int(load().mcs_launch_count())


def resize_linear_u8(src_ptr, src_w, src_h, src_pitch, src_frame_stride, dst_ptr, dst_w, dst_h, dst_pitch,
                     dst_frame_stride, channels, n_frames, stream=0):
    """``cv2.resize(..., INTER_LINEAR)`` of ``n_frames`` uint8 device images (include/mcs.h)."""
    check(load().mcs_resize_linear_u8(_vp(int(src_ptr)), int(src_w), int(src_h), int(src_pitch),
                                      int(src_frame_stride), _vp(int(dst_ptr)), int(dst_w), int(dst_h),
                                      int(dst_pitch), int(dst_frame_stride), int(channels), int(n_frames),
                                      _vp(int(stream))), "mcs_resize_linear_u8")


def copy_window_u8(dst_ptr, dst_pitch, dst_frame_stride, src_ptr, src_pitch, src_frame_stride, x_byte0, width_bytes,
                   y0, rows, n_frames, stream=0):
    """Window copy between two frame buffers of the same geometry (include/mcs.h)."""
    check(load().mcs_copy_window_u8(_vp(int(dst_ptr)), int(dst_pitch), int(dst_frame_stride), _vp(int(src_ptr)),
                                    int(src_pitch), int(src_frame_stride), int(x_byte0), int(width_bytes), int(y0),
                                    int(rows), int(n_frames), _vp(int(stream))), "mcs_copy_window_u8")


def upload_pageable_u8(windows, piece_bytes, threads, stream=0):
    """``windows``: (dst_ptr, src_ptr, staging_ptr, pitch, src_pitch, x_byte0, y0, width_bytes, rows) tuples
    (include/mcs.h: mcs_upload_pageable_u8).  The GIL is released for the duration of the call."""
    n = len(windows)
    if n == 0:
        return
    arr = ctypes.c_void_p * n
    dst = arr(*[int(w[0]) for w in windows])
    src = arr(*[int(w[1]) for w in windows])
    stg = arr(*[int(w[2]) for w in windows])
    pitch = np.array([w[3] for w in windows], dtype=np.int64)
    spitch = np.array([w[4] for w in windows], dtype=np.int64)
    xywh = np.array([w[5:9] for w in windows], dtype=np.int64).reshape(-1)
    check(load().mcs_upload_pageable_u8(n, dst, src, stg, pitch.ctypes.data_as(_c_i64p), spitch.ctypes.data_as(_c_i64p),
                                        xywh.ctypes.data_as(_c_i64p), int(piece_bytes), int(threads), _vp(int(stream))),
          "mcs_upload_pageable_u8")


def refit_homography(pts_a, pts_b, mask, h0, lm_iters=10):
    """Inlier refit + LM polish of a RANSAC winner on the host (include/mcs.h: mcs_refit_homography).
    ``pts_a`` / ``pts_b``: float32 N x 2, ``mask``: uint8 N or None, ``h0``: 3 x 3.  Returns H 3 x 3 float64."""
    a = np.ascontiguousarray(pts_a, dtype=np.float32).reshape(-1, 2)
    b = np.ascontiguousarray(pts_b, dtype=np.float32).reshape(-1, 2)
    if len(a) != len(b):
        raise ValueError("point sets differ in length: %d and %d" % (len(a), len(b)))
    m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8).reshape(-1)
    if m is not None and len(m) != len(a):
        raise ValueError("mask length %d for %d points" % (len(m), len(a)))
    h = np.ascontiguousarray(h0, dtype=np.float64).reshape(9)
    out = np.empty(9, dtype=np.float64)
    check(load().mcs_refit_homography(_vp(a.ctypes.data), _vp(b.ctypes.data), _vp(m.ctypes.data if m is not None else 0),
                                      len(a), _vp(h.ctypes.data), int(lm_iters), _vp(out.ctypes.data)),
          "mcs_refit_homography")
    return out.reshape(3, 3)


def _i32(a):
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(_c_i32p)


class Plan(object):
    """Owning wrapper of an ``mcs_plan*``."""

    def __init__(self, layer_kind, src_hw, fwd_h, origin_xy, rect_xyxy, out_w, out_h, channels, maps=None):
        """``maps``: optional list, one entry per layer: ``None`` or the ``(xy, frac)`` fixed-point
        map pair of a REMAP layer (int16 H x W x 2, uint16 H x W or None)."""
        lib = load()
        n = len(layer_kind)
        kind, kind_p = _i32(layer_kind)
        hw, hw_p = _i32(np.reshape(src_hw, (n, 2)))
        org, org_p = _i32(np.reshape(origin_xy, (n, 2)))
        rect, rect_p = _i32(np.reshape(rect_xyxy, (n, 4)))
        h = np.ascontiguousarray(np.reshape(fwd_h, (n, 9)), dtype=np.float64)
        handle = _vp()
        if maps is None or all(m is None for m in maps):
            check(lib.mcs_plan_create(ctypes.byref(handle), n, int(channels), kind_p, hw_p,
                                      h.ctypes.data_as(_c_f64p), org_p, rect_p, int(out_w), int(out_h)),
                  "mcs_plan_create")
        else:
            keep = []   # host arrays must outlive the call
            xy_p = (_vp * n)()
            fr_p = (_vp * n)()
            mhw = np.zeros((n, 2), dtype=np.int32)
            for k, m in enumerate(maps):
                if m is None:
                    continue
                xy = np.ascontiguousarray(m[0], dtype=np.int16)
                if xy.ndim != 3 or xy.shape[2] != 2:
                    raise ValueError("layer %d: map_xy must be H x W x 2 int16, got %r" % (k, xy.shape))
                keep.append(xy)
                xy_p[k] = xy.ctypes.data
                mhw[k] = xy.shape[:2]
                if m[1] is not None:
                    fr = np.ascontiguousarray(m[1], dtype=np.uint16)
                    if fr.shape != xy.shape[:2]:
                        raise ValueError("layer %d: map_frac shape %r != %r" % (k, fr.shape, xy.shape[:2]))
                    keep.append(fr)
                    fr_p[k] = fr.ctypes.data
            check(lib.mcs_plan_create_maps(ctypes.byref(handle), n, int(channels), kind_p, hw_p,
                                           h.ctypes.data_as(_c_f64p), org_p, rect_p, int(out_w), int(out_h),
                                           xy_p, fr_p, mhw.ctypes.data_as(_c_i32p)),
                  "mcs_plan_create_maps")
        self._h = handle
        self.n_layers = n
        self.channels = int(channels)
        self.out_w = int(out_w)
        self.out_h = int(out_h)
        self.src_hw = hw.copy()
        self._owned = None
        self.camera_weighted = False   # set_camera_weights is in force
        self.multiband = False         # set_multiband is in force
        self.blend_bands = 0           # its effective band count

    def close(self):
        if getattr(self, "_h", None) is not None and _lib is not None:
            _lib.mcs_plan_destroy(self._h)
        self._h = None

    __del__ = close

    def stitch(self, src_ptrs, src_pitch, src_frame_stride, n_frames, dst_ptr, dst_pitch,
               dst_frame_stride, stream=0):
        n = self.n_layers
        ptrs = (_vp * n)(*[int(p) for p in src_ptrs])
        pitch = (ctypes.c_int64 * n)(*[int(p) for p in src_pitch])
        fstr = (ctypes.c_int64 * n)(*[int(p) for p in src_frame_stride])
        check(_lib.mcs_stitch_u8(self._h, ptrs, pitch, fstr, int(n_frames), _vp(int(dst_ptr)),
                                 int(dst_pitch), int(dst_frame_stride), _vp(int(stream))),
              "mcs_stitch_u8")

    def owned_pixels(self, stream=0):
        """Per-layer owned-pixel counts (cached)."""
        if self._owned is None:
            out = (ctypes.c_int64 * MCS_MAX_LAYERS)()
            check(_lib.mcs_plan_owned_pixels(self._h, out, _vp(int(stream))), "mcs_plan_owned_pixels")
            self._owned = [int(out[k]) for k in range(self.n_layers)]
        return list(self._owned)

    def source_windows(self):
        """Per layer ``(x0, y0, x1, y1)``: the source pixels the layer's owned output pixels read."""
        out = (ctypes.c_int32 * (4 * self.n_layers))()
        check(_lib.mcs_plan_source_windows(self._h, out), "mcs_plan_source_windows")
        return [tuple(int(out[4 * k + j]) for j in range(4)) for k in range(self.n_layers)]

    def source_spans(self, layer, band_rows):
        """``[(x0, x1), ...]`` per band of ``band_rows`` source rows of ``layer``."""
        n = (int(self.src_hw[layer][0]) + band_rows - 1) // band_rows
        out = (ctypes.c_int32 * (2 * n))()
        check(_lib.mcs_plan_source_spans(self._h, int(layer), int(band_rows), out), "mcs_plan_source_spans")
        return [(int(out[2 * b]), int(out[2 * b + 1])) for b in range(n)]

    def algorithmic_bytes(self, stream=0):
        """SURVEY.md section 8(d): every output byte written once + one source
        byte per non-background output byte."""
        return self.out_w * self.out_h * self.channels + self.channels * sum(self.owned_pixels(stream))

    def last_variant(self):
        return int(_lib.mcs_plan_last_variant(self._h))

    def force_variant(self, variant):
        """0 = automatic, 1 = gather kernel, 2 = tiled (TMA-staged) kernel."""
        check(_lib.mcs_plan_force_variant(self._h, int(variant)), "mcs_plan_force_variant")

    def rows_need_padding(self):
        return bool(_lib.mcs_plan_rows_need_padding(self._h))

    def promise_padded_rows(self, promised=True):
        check(_lib.mcs_plan_promise_padded_rows(self._h, int(bool(promised))), "mcs_plan_promise_padded_rows")

    def set_feather(self, feather_log2):
        check(_lib.mcs_plan_set_feather(self._h, int(feather_log2)), "mcs_plan_set_feather")

    def set_blend(self, feather_log2, paste=None, weight_maps=None):
        """``paste``: ``[n_layers, 4]`` int32 or None; ``weight_maps``: list of n_layers optional 2-D uint8 arrays
        (entry k = weights of the paste of stage k over layer k-1's pasted rectangle) or None."""
        n = self.n_layers
        p_ptr = None
        if paste is not None:
            paste = np.ascontiguousarray(paste, dtype=np.int32).reshape(n, 4)
            p_ptr = paste.ctypes.data_as(_c_i32p)
        m_ptr, pitch_ptr, keep = None, None, []
        if weight_maps is not None and any(m is not None for m in weight_maps):
            if len(weight_maps) != n:
                raise ValueError("weight_maps must list %d entries (one per layer, entry 0 unused)" % n)
            ptrs = (ctypes.c_void_p * n)()
            pitches = np.zeros(n, np.int64)
            for k, m in enumerate(weight_maps):
                if m is None:
                    continue
                m = np.ascontiguousarray(m, dtype=np.uint8)
                if m.ndim != 2:
                    raise ValueError("weight map %d must be 2-D" % k)
                keep.append(m)
                ptrs[k] = m.ctypes.data
                pitches[k] = m.strides[0]
            m_ptr, pitch_ptr = ptrs, pitches.ctypes.data_as(_c_i64p)
            keep.append(pitches)
        check(_lib.mcs_plan_set_blend(self._h, int(feather_log2), p_ptr, m_ptr, pitch_ptr), "mcs_plan_set_blend")

    def set_camera_weights(self, weight_maps):
        """``weight_maps``: None (the plain overwrite) or a list of n_layers entries, each None (255 everywhere)
        or a uint8 array of that layer's source (height, width): the camera-weighted blend (include/mcs.h)."""
        n = self.n_layers
        self.multiband, self.blend_bands = False, 0   # every call switches the multi-band blend off
        if weight_maps is None:
            check(_lib.mcs_plan_set_camera_weights(self._h, None, None), "mcs_plan_set_camera_weights")
            self._owned = None
            self.camera_weighted = False
            return
        if len(weight_maps) != n:
            raise ValueError("weight_maps must list %d entries (one per layer)" % n)
        ptrs = (ctypes.c_void_p * n)()
        pitches = np.zeros(n, np.int64)
        keep = []   # host arrays must outlive the call
        for k, m in enumerate(weight_maps):
            if m is None:
                continue
            m = np.ascontiguousarray(m, dtype=np.uint8)
            if m.shape != tuple(int(v) for v in self.src_hw[k]):
                raise ValueError("weight map %d has shape %r, its source is %r" % (k, m.shape, tuple(self.src_hw[k])))
            keep.append(m)
            ptrs[k] = m.ctypes.data
            pitches[k] = m.strides[0]
        self._owned = None
        # on failure the library leaves the plan in the overwrite
        self.camera_weighted = False
        check(_lib.mcs_plan_set_camera_weights(self._h, ptrs, pitches.ctypes.data_as(_c_i64p)),
              "mcs_plan_set_camera_weights")
        self.camera_weighted = True

    def set_multiband(self, num_bands):
        """The multi-band blend of the camera weights (include/mcs.h mcs_plan_set_multiband); 0 switches it
        off.  Returns the effective band count."""
        self.multiband, self.blend_bands = False, 0
        check(_lib.mcs_plan_set_multiband(self._h, int(num_bands)), "mcs_plan_set_multiband")
        self.multiband = int(num_bands) > 0
        self.blend_bands = int(_lib.mcs_plan_multiband_bands(self._h))
        return self.blend_bands

    def tiled_ctas_per_sm(self):
        return int(_lib.mcs_plan_tiled_ctas_per_sm(self._h))

    def tiled_stats(self):
        """Work table of the tiled variant: tile counts per class, general passes, box bytes, frame block."""
        out = np.zeros(12, np.int32)
        check(_lib.mcs_plan_tiled_stats(self._h, out.ctypes.data_as(_c_i32p)), "mcs_plan_tiled_stats")
        keys = ("tiles", "fast", "warp", "copy", "zero", "fast_passes", "box_bytes", "frame_block", "band",
                "band_fused")
        return dict(zip(keys, (int(v) for v in out)))

    def tiled_status(self):
        """'' when the tiled variant is available, else why it is not."""
        return _lib.mcs_plan_tiled_status(self._h).decode(errors="replace")
