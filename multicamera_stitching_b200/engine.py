"""Host side of the fused compositing path: plan cache, device staging and the
calls into ``libmcs_b200.so``.

PyTorch is used here only as plumbing - device memory, pinned host memory,
streams.  All arithmetic happens in the sm_100a kernels behind the C ABI; if
the library or a CUDA device is missing the calls raise, there is no CPU path.
"""
import os
import threading
import weakref

import numpy as np
import torch

from . import _cabi
from .plan import PlanUnsupported, flatten_chain, plan_maps, plan_paste, plan_tables, stage_signature


def _stage_field(st, name):
    return st[name] if isinstance(st, dict) else getattr(st, name)


def _round_up(v, m):
    return (v + m - 1) // m * m


def _stage_threads():
    """Host threads that copy pageable frames into the pinned staging buffers (``$MCS_UPLOAD_THREADS``, default 4)."""
    return max(1, int(os.environ.get("MCS_UPLOAD_THREADS", "4")))


class PinnedResults(object):
    """Pinned host buffers for the panoramas handed back as ``numpy`` arrays.

    The reference returns a freshly allocated array per call (cv2 allocates it, StitcherClass.py:239);
    a download into fresh pageable memory costs three times what the same download into pinned memory
    does (1.39 ms against 0.46 ms for config 2's 25 MB, ``scripts/probe_single_call.py``).  So the
    array handed out is backed by a pinned buffer of this pool and the buffer comes back only when the
    array and every view of it have been garbage collected: two results never alias.  Callers that
    keep many panoramas alive exhaust the budget (``$MCS_PINNED_RESULT_BYTES``, default 512 MiB) and
    get ordinary pageable arrays from then on."""

    def __init__(self, budget=None):
        self.budget = int(os.environ.get("MCS_PINNED_RESULT_BYTES", str(512 << 20))) if budget is None else int(budget)
        self._free = {}     # shape -> [pinned tensors]
        self._bytes = 0     # pinned bytes allocated, handed out or free
        # re-entrant: a garbage collection that starts inside take() may finalise a result array on this very thread
        self._lock = threading.RLock()

    def take(self, shape):
        """A pinned uint8 tensor of this shape, or None when the budget is spent."""
        shape = tuple(int(v) for v in shape)
        n = int(np.prod(shape, dtype=np.int64))
        with self._lock:
            lst = self._free.get(shape)
            if lst:
                return lst.pop()
            if self._bytes + n > self.budget:     # drop free buffers of other shapes first
                for other in [k for k in self._free if k != shape]:
                    for t in self._free.pop(other):
                        self._bytes -= t.numel()
            if n == 0 or self._bytes + n > self.budget:
                return None
            self._bytes += n
        try:
            return self._alloc(shape)
        except RuntimeError:
            with self._lock:
                self._bytes -= n
            return None

    @staticmethod
    def _alloc(shape):
        return torch.empty(shape, dtype=torch.uint8, pin_memory=True)

    def give_back(self, t):
        with self._lock:
            self._free.setdefault(tuple(t.shape), []).append(t)

    def as_array(self, t):
        """``t`` as a numpy array; ``t`` returns to the pool when the array (and its views) are gone."""
        arr = t.numpy()
        weakref.finalize(arr, self.give_back, t).atexit = False
        return arr


class CompiledPlan(object):
    """A flattened chain plus its ``mcs_plan`` on one device."""

    def __init__(self, flat, device, feather_log2=0, blend_weights=None, camera_weights=None, blend_bands=0,
                 voronoi_seams=False, graphcut_frames=None, exposure_gains=None):
        self.flat = flat
        self.device = torch.device(device)
        self.feather_log2 = int(feather_log2)
        with torch.cuda.device(self.device):
            kind, src_hw, fwd, origin, rect = plan_tables(flat)
            self.handle = _cabi.Plan(kind, src_hw, fwd, origin, rect, flat.out_w, flat.out_h, flat.channels,
                                     maps=plan_maps(flat))
            maps = None
            if blend_weights is not None and any(w is not None for w in blend_weights):
                # stage s pastes over camera s + 1's warp: its map belongs to the layer of that camera
                maps = [None] * len(flat.layers)
                for k, l in enumerate(flat.layers):
                    if l.cam >= 1 and l.cam - 1 < len(blend_weights):
                        maps[k] = blend_weights[l.cam - 1]
            if self.feather_log2 or maps is not None:
                # the paste rectangles matter only when a super-mode crop cut a visible one
                self.handle.set_blend(self.feather_log2, plan_paste(flat), maps)
            if camera_weights is not None:   # one map per camera, in the layer order of the plan
                try:
                    self.handle.set_camera_weights([camera_weights[l.cam] if l.cam < len(camera_weights) else None
                                                    for l in flat.layers])
                except _cabi.McsError as e:
                    # more than 4 cameras meet at a pixel: the single-band kernel refuses the rig, the
                    # multi-band blend takes it (the library keeps the maps for it)
                    if not blend_bands or e.code != _cabi.MCS_ERR_UNSUPPORTED:
                        raise
                if blend_bands:
                    self.handle.set_multiband(blend_bands)
                if voronoi_seams:
                    try:
                        self.handle.set_voronoi_seams(True)
                    except _cabi.McsError as e:
                        if e.code == _cabi.MCS_ERR_UNSUPPORTED:
                            raise PlanUnsupported(str(e))
                        raise
                if exposure_gains is not None:   # before the graph-cut seams: they are found on compensated samples
                    self.handle.set_exposure_gains([exposure_gains[l.cam] for l in flat.layers])
                if graphcut_frames is not None:
                    self._find_graphcut_seams(graphcut_frames)
            # rows that are not a multiple of 4 bytes: run() always passes them through its
            # zero-padded scratch buffers, which is what the tiled kernel needs to serve them
            self.pad_rows = self._tiled() and self.handle.rows_need_padding()
            if self.pad_rows:
                self.handle.promise_padded_rows(True)
        self.cams = [l.cam for l in flat.layers]
        self.out_w, self.out_h, self.channels = flat.out_w, flat.out_h, flat.channels

    def _upload_frame_set(self, frames_by_cam, what):
        """One host frame-set (``frames_by_cam[c]``: H x W x 3 uint8) on the device: ``{cam: tensor}``."""
        dev = {}
        for l in self.flat.layers:
            f = np.asarray(frames_by_cam[l.cam])
            want = tuple(l.src_hw) + (3,)
            if f.dtype != np.uint8 or f.shape != want:
                raise ValueError("%s: camera %d's frame is %s %r, the plan needs uint8 %r"
                                 % (what, l.cam, f.dtype, f.shape, want))
            if l.cam not in dev:
                dev[l.cam] = torch.from_numpy(np.array(f)).to(self.device)
        return dev

    def estimate_gains(self, frames_by_cam):
        """The exposure gains of one host frame-set (include/mcs.h mcs_plan_estimate_gains), per camera
        (``{cam: gain}``).  The plan is unchanged."""
        with torch.cuda.device(self.device):
            dev = self._upload_frame_set(frames_by_cam, "exposure gains")
            gains = self.handle.estimate_gains([dev[l.cam].data_ptr() for l in self.flat.layers],
                                               [dev[l.cam].stride(0) for l in self.flat.layers])
        return {l.cam: float(g) for l, g in zip(self.flat.layers, gains)}

    def _find_graphcut_seams(self, frames_by_cam):
        """Upload one host frame-set (``frames_by_cam[c]``: H x W x 3 uint8), find the graph-cut seams on it
        (include/mcs.h mcs_plan_set_graphcut_seams) and drop the upload."""
        dev = self._upload_frame_set(frames_by_cam, "graph-cut seams")
        try:
            self.handle.set_graphcut_seams([dev[l.cam].data_ptr() for l in self.flat.layers],
                                           [dev[l.cam].stride(0) for l in self.flat.layers])
        except _cabi.McsError as e:
            if e.code == _cabi.MCS_ERR_UNSUPPORTED:
                raise PlanUnsupported(str(e))
            raise

    def _tiled(self):
        """Whether the tiled kernel serves this plan (it does not serve the camera-weighted blends)."""
        return self.handle.tiled_status() == "" and not (self.handle.camera_weighted or self.handle.multiband)

    # ---- geometry helpers -------------------------------------------------
    def out_shape(self, n_frames=None):
        s = (self.out_h, self.out_w) + ((self.channels,) if self.flat.ndim == 3 else ())
        return s if n_frames is None else (n_frames,) + s

    def algorithmic_bytes(self):
        with torch.cuda.device(self.device):
            return self.handle.algorithmic_bytes(torch.cuda.current_stream().cuda_stream)

    def owned_pixels(self):
        with torch.cuda.device(self.device):
            return self.handle.owned_pixels(torch.cuda.current_stream().cuda_stream)

    # ---- what the host has to send ------------------------------------------
    BAND = int(os.environ.get("MCS_UPLOAD_BAND", "64"))   # source rows per upload band

    def upload_bands(self, whole=False):
        """Per camera, the byte windows of a frame that can reach the panorama: a list of copies
        ``{b0, nbytes, y0, rows}`` (bytes ``[b0, b0 + nbytes)`` of rows ``[y0, y0 + rows)``), from
        ``mcs_plan_source_spans`` per band of ``BAND`` source rows, columns widened to 64-byte
        boundaries, neighbouring bands with the same range merged.  What lies under the pasted
        inner canvas (StitcherClass.py:240-241) is never read by the kernels, so a host-facing
        caller need not upload it.  Returns ``{cam: (row_bytes, rows, copies)}``; ``whole=True``
        (and feather mode) lists whole frames."""
        key = bool(whole)
        cache = self.__dict__.setdefault("_bands", {})
        if key not in cache:
            out = {}
            for k, l in enumerate(self.flat.layers):
                h, w = int(l.src_hw[0]), int(l.src_hw[1])
                px = self.channels
                row = w * px
                copies = []
                spans = [(0, w)] * (-(-h // self.BAND)) if whole else self.handle.source_spans(k, self.BAND)
                for b, (x0, x1) in enumerate(spans):
                    if x1 <= x0:
                        continue
                    b0 = (x0 * px) // 64 * 64
                    b1 = min(row, -(-(x1 * px) // 64) * 64)
                    y0, rows = b * self.BAND, min(self.BAND, h - b * self.BAND)
                    last = copies[-1] if copies else None
                    if last and last["b0"] == b0 and last["nbytes"] == b1 - b0 and last["y0"] + last["rows"] == y0:
                        last["rows"] += rows
                    else:
                        copies.append(dict(b0=b0, nbytes=b1 - b0, y0=y0, rows=rows))
                out[l.cam] = (row, h, copies)
            cache[key] = out
        return cache[key]

    # ---- launch -----------------------------------------------------------
    def _describe(self, t, batched):
        """(data_ptr, pitch_bytes, frame_stride_bytes) of a uint8 CUDA tensor
        holding [F,]H,W[,C] frames with dense pixels."""
        if t.dtype != torch.uint8 or not t.is_cuda:
            raise TypeError("frames must be uint8 CUDA tensors, got %s on %s" % (t.dtype, t.device))
        nd = self.flat.ndim + (1 if batched else 0)
        if t.dim() != nd:
            raise ValueError("expected a %d-D frame tensor, got shape %r" % (nd, tuple(t.shape)))
        st = t.stride()
        if self.flat.ndim == 3:
            dense = st[-1] == 1 and st[-2] == self.channels
            pitch = st[-3]
        else:
            dense = st[-1] == 1
            pitch = st[-2]
        if not dense:
            raise ValueError("frame pixels must be densely packed (strides %r)" % (st,))
        return t.data_ptr(), pitch, (st[0] if batched else 0)

    def _realigned(self, cam, t, p, pitch, fs, F, batched, stream):
        h, w = int(t.shape[-3 if self.flat.ndim == 3 else -2]), int(t.shape[-2 if self.flat.ndim == 3 else -1])
        row = w * self.channels
        pitch16 = _round_up(row, 16)
        scratch = self.__dict__.setdefault("_scratch", {})
        buf = scratch.get(cam)
        if buf is None or buf.shape[0] < F or buf.shape[1:] != (h, pitch16) or buf.device != t.device:
            buf = torch.zeros((F, h, pitch16), dtype=torch.uint8, device=t.device)
            scratch[cam] = buf
        with torch.cuda.device(self.device):
            s = torch.cuda.current_stream() if stream is None else stream
            _cabi.copy_window_u8(buf.data_ptr(), pitch16, h * pitch16, p, pitch, fs if batched and F > 1 else h * pitch,
                                 0, row, 0, h, F, s.cuda_stream)
        return buf.data_ptr(), pitch16, h * pitch16

    def new_output(self, n_frames=None, pitch_align=1):
        """Uninitialised output tensor (every byte of it is written by the
        kernel).  With ``pitch_align`` > 1 rows are padded and a strided view
        is returned."""
        F = 1 if n_frames is None else n_frames
        row = self.out_w * self.channels
        pitch = _round_up(max(row, 1), pitch_align)
        buf = torch.empty((F, self.out_h, pitch), dtype=torch.uint8, device=self.device)
        if self.flat.ndim == 3:
            view = torch.as_strided(buf, (F, self.out_h, self.out_w, self.channels),
                                    (self.out_h * pitch, pitch, self.channels, 1))
        else:
            view = torch.as_strided(buf, (F, self.out_h, self.out_w), (self.out_h * pitch, pitch, 1))
        return view if n_frames is not None else view[0]

    def run(self, frames_by_cam, out=None, n_frames=None, stream=None):
        """Composite.  ``frames_by_cam[c]`` is the CUDA tensor of camera ``c``
        ([H,W,C] or, when ``n_frames`` is given, [F,H,W,C]).  Returns ``out``."""
        batched = n_frames is not None
        F = n_frames if batched else 1
        if out is None:
            out = self.new_output(n_frames)
        if tuple(out.shape) != self.out_shape(n_frames):
            raise ValueError("output shape %r != %r" % (tuple(out.shape), self.out_shape(n_frames)))
        ptrs, pitches, fstrides = [], [], []
        tiled = self._tiled()
        for l in self.flat.layers:
            t = frames_by_cam[l.cam]
            want = ((F,) if batched else ()) + tuple(l.src_hw) + ((self.channels,) if self.flat.ndim == 3 else ())
            if tuple(t.shape) != want:
                raise ValueError("camera %d: frame shape %r != %r" % (l.cam, tuple(t.shape), want))
            p, pitch, fs = self._describe(t, batched)
            if tiled and (self.pad_rows or p % 16 or pitch % 16 or (batched and F > 1 and fs % 16)):
                # The TMA-staged kernel needs 16-byte aligned rows; the gather kernel that would
                # serve this layout is ~5x slower, so the frames take one extra device-side pass
                # into a pitched scratch buffer (plain cudaMemcpy3DAsync) instead.
                p, pitch, fs = self._realigned(l.cam, t, p, pitch, fs, F, batched, stream)
            ptrs.append(p)
            pitches.append(pitch)
            fstrides.append(fs)
        dp, dpitch, dfs = self._describe(out, batched)
        with torch.cuda.device(self.device):
            s = torch.cuda.current_stream() if stream is None else stream
            self.handle.stitch(ptrs, pitches, fstrides, F, dp, dpitch, dfs, s.cuda_stream)
        return out


class CompositeEngine(object):
    """Plan cache + host<->device staging for one ``Stitcher``."""

    STAGE_PIECE_BYTES = 1 << 20   # staging granularity of upload_frames

    def __init__(self, device=None):
        self._device = device
        self._plans = {}          # insertion-ordered: least recently used first
        self.max_plans = 16
        self._staging = {}
        self._pinned_in = {}      # (cam, shape) -> [pinned tensor, event of its last DMA, frame being staged]
        self.results = PinnedResults()

    @property
    def device(self):
        if self._device is None:
            if not torch.cuda.is_available():
                raise _cabi.McsError("no CUDA device: the compositing path has no CPU fallback")
            self._device = torch.device("cuda", torch.cuda.current_device())
        return torch.device(self._device)

    def plan_for(self, stages, cam_shapes, device=None, feather_log2=0, blend_weights=None, camera_weights=None,
                 blend_bands=0, voronoi_seams=False, graphcut_seams=None, exposure_gains=None):
        """Compiled plan for this chain state and these frame shapes, or None
        when no stage is calibrated (decided on the host, no device needed).  ``graphcut_seams``: None or
        ``(digest, frames by camera)`` of the frame-set the graph-cut seams are found on; ``exposure_gains``: None
        or a tuple of gains by camera."""
        shapes = tuple(tuple(int(v) for v in s) for s in cam_shapes)
        sig = tuple(stage_signature(st) for st in stages)
        if all(s is None for s in sig):
            return None
        device = torch.device(device) if device is not None else self.device
        feather_log2 = int(feather_log2 or 0)
        wkey = None
        if blend_weights is not None and any(w is not None for w in blend_weights):
            wkey = tuple(None if w is None else (np.asarray(w).shape, hash(np.ascontiguousarray(w, dtype=np.uint8).tobytes()))
                         for w in blend_weights)
        ckey = None
        if camera_weights is not None:
            ckey = tuple(None if w is None else (np.asarray(w).shape, hash(np.ascontiguousarray(w, dtype=np.uint8).tobytes()))
                         for w in camera_weights)
        blend_bands = int(blend_bands or 0)
        voronoi_seams = bool(voronoi_seams)
        gkey = None if graphcut_seams is None else graphcut_seams[0]
        ekey = None if exposure_gains is None else tuple(float(g) for g in exposure_gains)
        key = (str(device), shapes, sig, feather_log2, wkey, ckey, blend_bands, voronoi_seams, gkey, ekey)
        if key in self._plans:
            self._plans[key] = self._plans.pop(key)      # most recently used last
        else:
            flat = flatten_chain(stages, shapes)
            while len(self._plans) >= self.max_plans:     # evict the least recently used, one at a time
                self._plans.pop(next(iter(self._plans)))
            self._plans[key] = (CompiledPlan(flat, device, feather_log2, blend_weights, camera_weights, blend_bands,
                                             voronoi_seams, None if graphcut_seams is None else graphcut_seams[1],
                                             ekey)
                                if flat is not None else None)
        return self._plans[key]

    def upload(self, cam, arr, device, bands=None):
        """Host frame -> (reused) device tensor on the current stream.  ``bands`` =
        ``CompiledPlan.upload_bands()[cam]``: only those byte windows of the frame are sent, the
        rest of the device tensor keeps whatever it held (the kernels never read it)."""
        t = torch.from_numpy(np.ascontiguousarray(arr)) if isinstance(arr, np.ndarray) else arr.contiguous()
        if t.dtype != torch.uint8:
            raise TypeError("frames must be uint8, got %s" % (t.dtype,))
        key = (cam, tuple(t.shape), str(device))
        buf = self._staging.get(key)
        if buf is None:
            buf = torch.empty(t.shape, dtype=torch.uint8, device=device)
            self._staging[key] = buf
        if bands is not None:
            row, h, copies = bands
            whole = len(copies) == 1 and copies[0]["nbytes"] == row and copies[0]["rows"] == h
            if not whole and t.dim() in (2, 3) and int(t.shape[0]) == h and t.numel() == row * h:
                stream = torch.cuda.current_stream().cuda_stream
                for w in copies:
                    _cabi.copy_window_u8(buf.data_ptr(), row, row * h, t.data_ptr(), row, row * h, w["b0"], w["nbytes"],
                                         w["y0"], w["rows"], 1, stream)
                return buf
        buf.copy_(t, non_blocking=True)
        return buf

    def upload_frames(self, cams, frames, device, bands=None):
        """Host frames of one frame-set -> device tensors, ``{cam: tensor}``.  ``numpy`` frames are
        pageable memory: ``mcs_upload_pageable_u8`` copies what the panorama can see of each camera
        (``bands[cam]``) into per-camera pinned buffers with a few host threads, in pieces of about
        ``STAGE_PIECE_BYTES``, and issues every piece's DMA as soon as it has landed - instead of the
        driver staging the pageable copies one after the other (``scripts/probe_single_call.py``).
        Everything else goes through ``upload``."""
        out = {}
        windows = []
        ents = []
        for cam in cams:
            arr = frames[cam]
            b = None if bands is None else bands.get(cam)
            if not (isinstance(arr, np.ndarray) and arr.dtype == np.uint8 and arr.ndim in (2, 3) and arr.size):
                out[cam] = self.upload(cam, arr, device, b)
                continue
            shape = tuple(int(v) for v in arr.shape)
            h, row = shape[0], arr.size // shape[0]
            if arr.strides[0] < row or not arr[0].flags.c_contiguous:
                arr = np.ascontiguousarray(arr)     # rows must be dense; a row stride is fine
            ent = self._pinned_in.get((cam, shape))
            if ent is None:
                ent = self._pinned_in[(cam, shape)] = [torch.empty(shape, dtype=torch.uint8, pin_memory=True), None, None]
            elif ent[1] is not None:
                ent[1].synchronize()        # the DMAs of the previous call have read the buffer
            ent[2] = arr                    # keeps a converted copy alive until the call below returns
            ents.append(ent)
            key = (cam, shape, str(device))
            buf = self._staging.get(key)
            if buf is None:
                buf = self._staging[key] = torch.empty(shape, dtype=torch.uint8, device=device)
            out[cam] = buf
            if b is not None and b[0] == row and b[1] == h:
                copies = b[2]
            else:
                copies = [dict(b0=0, nbytes=row, y0=0, rows=h)]
            for w in copies:
                windows.append((buf.data_ptr(), arr.ctypes.data, ent[0].data_ptr(), row, arr.strides[0],
                                w["b0"], w["y0"], w["nbytes"], w["rows"]))
        if windows:
            stream = torch.cuda.current_stream()
            _cabi.upload_pageable_u8(windows, self.STAGE_PIECE_BYTES, _stage_threads(), stream.cuda_stream)
            for ent in ents:
                if ent[1] is None:
                    ent[1] = torch.cuda.Event()
                ent[1].record(stream)
                ent[2] = None
        return out

    def download(self, res):
        """Device panorama -> a new ``numpy`` array (blocking), through the pinned result pool."""
        host = self.results.take(res.shape)
        if host is None:
            host = torch.empty(res.shape, dtype=torch.uint8)
            host.copy_(res)  # synchronous D2H into a fresh pageable array, like cv2 allocating its result
            return host.numpy()
        host.copy_(res, non_blocking=True)
        torch.cuda.current_stream(res.device).synchronize()
        return self.results.as_array(host)

    def resize(self, t, hw, batched=False):
        """``cv2.resize(frame, (w, h), interpolation=cv2.INTER_LINEAR)`` of a uint8 CUDA tensor
        ([H,W[,C]] or, batched, [F,H,W[,C]]) into a new tensor: the shape fix-up of the
        reference's stitch (StitcherClass.py:226-233) through ``mcs_resize_linear_u8``."""
        if t.dtype != torch.uint8 or not t.is_cuda:
            raise TypeError("resize expects a uint8 CUDA tensor, got %s on %s" % (t.dtype, t.device))
        lead = 1 if batched else 0
        if t.dim() - lead not in (2, 3):
            raise ValueError("resize expects H x W or H x W x C frames, got shape %r" % (tuple(t.shape),))
        C = int(t.shape[lead + 2]) if t.dim() - lead == 3 else 1
        F = int(t.shape[0]) if batched else 1
        hs, ws = int(t.shape[lead]), int(t.shape[lead + 1])
        hd, wd = int(hw[0]), int(hw[1])
        st = t.stride()
        dense = st[-1] == 1 and (t.dim() - lead == 2 or st[-2] == C)
        if not dense or (batched and F > 1 and st[0] < 0):
            t = t.contiguous()
            st = t.stride()
        out = torch.empty(t.shape[:lead] + (hd, wd) + t.shape[lead + 2:], dtype=torch.uint8, device=t.device)
        with torch.cuda.device(t.device):
            _cabi.resize_linear_u8(t.data_ptr(), ws, hs, st[lead], st[0] if batched else 0,
                                   out.data_ptr(), wd, hd, wd * C, hd * wd * C, C, F,
                                   torch.cuda.current_stream().cuda_stream)
        return out

    def reset(self):
        self._plans.clear()
        self._staging.clear()
        self._pinned_in.clear()
