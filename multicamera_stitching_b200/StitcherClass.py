"""B200-native ``Stitcher`` / ``StitcherBase``.

Drop-in for the classes of the reference's
``PostScripts/Stitcher/StitcherClass.py`` (same class, method, argument and
attribute names, same return conventions and graceful-degradation behaviour),
re-implemented for Python 3 with the per-frame work moved onto the GPU:

* ``Stitcher.stitch`` (reference :114-136) no longer runs N-1 sequential
  ``cv2.warpPerspective`` + paste stages; the calibrated chain is flattened
  once into a compositing plan and every panorama is ONE launch of the fused
  warp+paste kernel behind ``mcs_stitch_u8`` (include/mcs.h).
* ``StitcherBase.matchKeypoints`` (reference :405-448) runs the brute-force
  Hamming 2-NN + ratio test and the RANSAC hypothesis scoring on the GPU
  (``mcs_match_hamming_top2`` / ``mcs_ransac_homography``).

Frames may be ``numpy`` arrays (result: a new ``numpy`` array, like the
reference) or uint8 CUDA tensors (result: a CUDA tensor, nothing leaves the
device).  There is no CPU fallback: without the CUDA library these methods
raise.
"""
import hashlib
import os
import pickle

import cv2
import numpy as np

from .extended_rospylogs import Debugger, DEBUG_LEVEL_0
from .Utils import get_projection_point_dst
from .plan import PlanUnsupported

# ---------------------------------------------------------------------------


def get_opencv_major_version(lib=None):
    """Major version number of OpenCV (reference :41-47)."""
    if lib is None:
        lib = cv2
    return int(lib.__version__.split(".")[0])


def is_cv3(or_better=False):
    """Reference :30-39."""
    major = get_opencv_major_version()
    return major >= 3 if or_better else major == 3


def _is_tensor(x):
    return type(x).__module__.startswith("torch") and hasattr(x, "is_cuda")


def _shape_of(img):
    return tuple(int(v) for v in img.shape)


# ---------------------------------------------------------------------------
class Stitcher(Debugger):
    """N-camera panorama: a chain of N-1 pairwise stitchers (reference :50-177)."""

    # Class-level default: an object unpickled from a configuration the REFERENCE saved is built without
    # __init__ and has no blend-mode attribute.
    feather_log2 = 0
    # Optional weight maps of the pastes (extension, include/mcs.h mcs_plan_set_blend): a list with one entry per
    # stage, None or a uint8 array of the shape of that stage's imageB (the running canvas) holding the canvas'
    # weight in units of 1 / 2**feather_log2; None everywhere = the distance ramp of feather_log2.
    blend_weights = None
    # Optional camera-weighted blend (extension, include/mcs.h mcs_plan_set_camera_weights): a dict
    # {label: None or a uint8 array of that camera's calibrated (h, w)} - every camera that sees a pixel
    # contributes, weighted by its own map and normalised by the summed weights; None = 255 everywhere, a
    # missing label likewise.  None (the default) keeps the reference's overwrite.  ``edge_ramp`` gives the
    # FeatherBlender-style map.
    camera_weights = None
    # Optional multi-band blend of the camera weights (extension, include/mcs.h mcs_plan_set_multiband): 0 (the
    # default) = off, 1..8 = the Laplacian-pyramid blend of OpenCV's MultiBandBlender with that many bands (clamped
    # to ceil(log2) of the panorama's longer side).  ``camera_weights`` supplies the masks; without them every camera
    # weighs 255 everywhere.
    blend_bands = 0
    # Optional Voronoi seams for the multi-band blend (extension, include/mcs.h mcs_plan_set_voronoi_seams): True cuts
    # every overlap at OpenCV's VoronoiSeamFinder seam before the blend, so that each overlap pixel takes its fine
    # detail from one camera and only the low bands mix across the seam.  Needs ``blend_bands`` > 0.
    voronoi_seams = False
    # Optional graph-cut seams for the multi-band blend (extension, include/mcs.h mcs_plan_set_graphcut_seams), set by
    # ``find_graphcut_seams``: None, or ``(digest, frames)`` - the read-only frame-set the seams are found on, in
    # camera order, and its digest, which keys the compiled plans.  Needs ``blend_bands`` > 0, not with
    # ``voronoi_seams``.
    graphcut_seams = None
    # Optional exposure compensation of the camera-weighted and multi-band blends (extension, include/mcs.h
    # mcs_plan_set_exposure_gains): None, or {label: gain} - every camera's sample v becomes saturate_u8(rint(v * gain))
    # before it is blended, as OpenCV's GainCompensator applies its gains; a missing label keeps gain 1.
    # ``compensate_exposure`` estimates them from a frame-set; they are plain floats, to read, set, pickle and reuse.
    # Needs ``camera_weights`` or ``blend_bands`` > 0.
    exposure_gains = None

    def __init__(self, images_dic, super_mode=False):
        # labels sorted like np.sort(images_dic.keys()) (reference :61)
        self.img_labels = np.sort(list(images_dic.keys()))
        self.stitcher_labels = []
        for idx in range(len(self.img_labels) - 1):
            left = self.img_labels[idx] if idx == 0 else self.stitcher_labels[-1]
            self.stitcher_labels.append("({}&{})".format(left, self.img_labels[idx + 1]))
        self.stitchers = [StitcherBase(sid=label, super_mode=super_mode)
                          for label in self.stitcher_labels]
        # Blend mode (extension; the reference only overwrites, :240-241): 0 = overwrite, n > 0 =
        # feather every paste over 2**n pixels (include/mcs.h mcs_plan_set_feather).
        self.feather_log2 = 0

    # -- engine plumbing (never pickled) -------------------------------------
    def _engine_(self):
        eng = self.__dict__.get("_engine")
        if eng is None:
            from .engine import CompositeEngine
            eng = CompositeEngine()
            self.__dict__["_engine"] = eng
        return eng

    def __getstate__(self):
        state = dict(self.__dict__)
        state.pop("_engine", None)
        return state

    # -- calibration ---------------------------------------------------------
    def calibrate_stitcher(self, images_dic, save=True, save_path=""):
        """Calibrate every pairwise stitcher on ``images_dic`` and optionally
        save the configuration (reference :77-112).  Stage ``k`` calibrates the
        next camera against the canvas stitched so far."""
        img_result = None
        for idx in range(len(self.img_labels) - 1):
            if idx == 0:
                images = (images_dic[self.img_labels[0]], images_dic[self.img_labels[1]])
            else:
                images = (img_result, images_dic[self.img_labels[idx + 1]])
            self.stitchers[idx].calibrate(images=images, ratio=0.75, reprojThresh=3.0,
                                          xoffset=0, yoffset=0)
            img_result = self.stitchers[idx].stitch(images=images)
        self._report()
        if save:
            self.save_stitcher(save_path)

    def calibrate_from_homographies(self, img_shapes, homographies, xoffset=0, yoffset=0):
        """Calibrate the chain from known homographies instead of matched
        features (extension used for fixed rigs and synthetic benchmarks).
        ``homographies[k]`` maps camera ``k+1`` into the canvas of stage
        ``k-1`` (camera 0's frame for ``k == 0``), i.e. it is what
        ``matchKeypoints`` would have returned at stage ``k``."""
        shapeB = tuple(img_shapes[0])
        for idx, H in enumerate(homographies):
            st = self.stitchers[idx]
            st.set_homography(H, shapeA=tuple(img_shapes[idx + 1]), shapeB=shapeB,
                              xoffset=xoffset, yoffset=yoffset)
            shapeB = st.result_shape()
        self.__dict__.pop("_engine", None)

    def _report(self):
        for st in self.stitchers:
            self.debugger(DEBUG_LEVEL_0, "[STITCHER]: {}".format(st),
                          log_type="err" if st.status is None else "info")

    # -- per-frame path --------------------------------------------------------
    def stitch(self, images_dic, draw_descriptors=False):
        """Stitched panorama of ``images_dic`` (reference :114-136)."""
        if len(images_dic) > len(self.img_labels):
            self.debugger(DEBUG_LEVEL_0, "[STITCHER] Images dictionary is bigger than list", log_type="warn")
        elif len(images_dic) < len(self.img_labels):
            self.debugger(DEBUG_LEVEL_0, "[STITCHER] Images dictionary is inferior to labels list",
                          log_type="err")
            return images_dic[self.img_labels[-1]]
        if len(self.img_labels) < 2:
            return images_dic[self.img_labels[-1]]
        frames = [images_dic[label] for label in self.img_labels]
        out = _composite(self._engine_(), self.stitchers, frames, batched=False, debugger=self,
                         feather_log2=getattr(self, "feather_log2", 0), blend_weights=self.blend_weights,
                         camera_weights=self._camera_weight_list(), blend_bands=self._blend_bands(),
                         voronoi_seams=self._voronoi_seams(), graphcut_seams=self._graphcut_seams(),
                         exposure_gains=self._exposure_gains())
        if draw_descriptors and not _is_tensor(out):
            out = self._draw_overlays(out, frames)
        return out

    def _draw_overlays(self, out, frames):
        """The reference draws every stage's overlay into the canvas that stage produced, before the optional
        crop (:244-251); the canvas is then pasted verbatim by the next stage, so in the final panorama the
        overlays lie on top of everything, earlier stages below later ones, each at its canvas' position and
        clipped to what is left of that canvas."""
        try:
            flat = self.plan([f.shape for f in frames]).flat
        except Exception:   # segmented chains (a resized canvas in between): only the last stage is in final coordinates
            flat = None
        if flat is None or (flat.out_h, flat.out_w) != tuple(out.shape[:2]):
            return self.stitchers[-1].draw_descriptors(img_src=out)
        by_cam = {l.cam: l for l in flat.layers}
        for s, st in enumerate(self.stitchers):
            if st.cachedAH is None or (s + 1) not in by_cam:
                continue
            l = by_cam[s + 1]
            x0, y0, x1, y1 = (int(v) for v in l.rect)
            if x1 <= x0 or y1 <= y0:
                continue
            # draw on the visible part of the stage's canvas plus a margin that is still canvas (anti-aliased text
            # next to the crop edge takes coverage from glyph parts beyond it; clipping at the canvas edge itself is
            # what the reference does too)
            m = 32
            cw, ch = int(st.ABSize[0]), int(st.ABSize[1])
            ex0, ey0 = max(x0 - m, l.ox), max(y0 - m, l.oy)
            ex1, ey1 = min(x1 + m, l.ox + cw), min(y1 + m, l.oy + ch)
            sub = np.zeros((ey1 - ey0, ex1 - ex0) + out.shape[2:], dtype=out.dtype)
            sub[y0 - ey0:y1 - ey0, x0 - ex0:x1 - ex0] = out[y0:y1, x0:x1]
            st._draw_descriptors_at(sub, offset=(l.ox - ex0, l.oy - ey0), canvas_size=st.ABSize)
            out[y0:y1, x0:x1] = sub[y0 - ey0:y1 - ey0, x0 - ex0:x1 - ex0]
        return out

    def stitch_batch(self, frames_dic, out=None):
        """Composite ``F`` frame-sets in one launch.  ``frames_dic[label]`` is a
        uint8 CUDA tensor ``[F, H, W, C]``; returns (or fills ``out``) a CUDA
        tensor ``[F, H_out, W_out, C]``.  Extension of the reference API."""
        frames = [frames_dic[label] for label in self.img_labels]
        return _composite(self._engine_(), self.stitchers, frames, batched=True, out=out, debugger=self,
                          feather_log2=getattr(self, "feather_log2", 0), blend_weights=self.blend_weights,
                          camera_weights=self._camera_weight_list(), blend_bands=self._blend_bands(),
                          voronoi_seams=self._voronoi_seams(), graphcut_seams=self._graphcut_seams(),
                          exposure_gains=self._exposure_gains())

    def plan(self, img_shapes, device=None):
        """Compiled plan (``engine.CompiledPlan``) for frames of these shapes."""
        return self._engine_().plan_for(self.stitchers, [tuple(s) for s in img_shapes], device,
                                        feather_log2=getattr(self, "feather_log2", 0), blend_weights=self.blend_weights,
                                        camera_weights=self._camera_weight_list(), blend_bands=self._blend_bands(),
                                        voronoi_seams=self._voronoi_seams(), graphcut_seams=self._graphcut_seams(),
                                        exposure_gains=self._exposure_gains())

    def _blend_bands(self):
        """``blend_bands`` checked: an int in 0..8."""
        n = self.blend_bands
        if isinstance(n, bool) or not isinstance(n, (int, np.integer)) or not 0 <= int(n) <= 8:
            raise ValueError("blend_bands must be an integer in 0..8, got %r" % (n,))
        return int(n)

    def _voronoi_seams(self):
        """``voronoi_seams`` checked: a bool, True only with ``blend_bands`` > 0."""
        v = self.voronoi_seams
        if not isinstance(v, (bool, np.bool_)):
            raise ValueError("voronoi_seams must be True or False, got %r" % (v,))
        if v and not self._blend_bands():
            raise ValueError("voronoi_seams cuts the masks of the multi-band blend: set blend_bands > 0 too")
        return bool(v)

    def find_graphcut_seams(self, images_dic):
        """Cut the multi-band blend's masks at graph-cut seams (OpenCV's ``GraphCutSeamFinder("COST_COLOR")``) found
        on this frame-set, ``{label: H x W x 3 uint8 frame}`` of every camera's calibrated size: each overlap is cut
        where the two cameras agree on colour, around objects they see at different parallax.  Keeps a read-only
        copy of the frames; the seams are found on the device when a plan is compiled and stay until this is called
        again (new frames find new seams) or with None (back to the full masks)."""
        if images_dic is None:
            self.graphcut_seams = None
            return
        frames = self._frame_set(images_dic, "find_graphcut_seams")
        digest = hashlib.sha256()
        for f in frames:
            digest.update(repr(f.shape).encode())
            digest.update(f.data)
        self.graphcut_seams = (digest.hexdigest(), tuple(frames))

    def _frame_set(self, images_dic, what):
        """Read-only copies, in camera order, of one frame-set ``{label: H x W x 3 uint8 frame}`` of every camera's
        calibrated size."""
        labels = [str(l) for l in self.img_labels]
        by_label = {str(k): v for k, v in dict(images_dic).items()}
        missing = sorted(set(labels) - set(by_label))
        if missing:
            raise ValueError("%s needs a frame of every camera, missing %r" % (what, missing))
        frames = []
        for i, label in enumerate(labels):
            f = by_label[label]
            if _is_tensor(f):
                f = f.detach().cpu().numpy()
            f = np.asarray(f)
            st = self.stitchers[max(0, i - 1)]
            size = st.BimgSize if i == 0 else st.AimgSize
            want = None if size is None else tuple(size[:2]) + (3,)
            if f.dtype != np.uint8 or f.ndim != 3 or f.shape[2] != 3 or (want is not None and f.shape != want):
                raise ValueError("%s: camera %r needs a uint8 frame of its calibrated (h, w, 3) %r, got %s %r"
                                 % (what, label, want, f.dtype, f.shape))
            f = np.array(f, np.uint8, order="C", copy=True)
            f.setflags(write=False)
            frames.append(f)
        return frames

    def compensate_exposure(self, images_dic):
        """Estimate every camera's exposure gain on this frame-set, ``{label: H x W x 3 uint8 frame}`` of every camera's
        calibrated size, as OpenCV's ``GainCompensator`` does (on the device), store the gains in ``exposure_gains``
        and return them (``{label: gain}``).  Only pixels where two cameras' weights are both 255 count.  The gains
        stay until this is called again or with None (no compensation).  Needs ``camera_weights`` or
        ``blend_bands`` > 0."""
        if images_dic is None:
            self.exposure_gains = None
            return None
        frames = self._frame_set(images_dic, "compensate_exposure")
        cw = self._camera_weight_list()
        if cw is None:
            raise ValueError("exposure gains compensate the camera-weighted and multi-band blends: set camera_weights "
                             "or blend_bands > 0 too")
        # the gains are estimated on the uncut weights and uncompensated samples: a plan without seams or gains
        plan = self._engine_().plan_for(self.stitchers, [f.shape for f in frames], camera_weights=cw,
                                        blend_bands=self._blend_bands())
        if plan is None:
            raise ValueError("compensate_exposure needs a calibrated chain")
        by_cam = plan.estimate_gains(frames)
        self.exposure_gains = {str(label): by_cam.get(i, 1.0) for i, label in enumerate(self.img_labels)}
        return dict(self.exposure_gains)

    def _exposure_gains(self):
        """``exposure_gains`` checked and as a tuple of floats in camera order (missing labels 1), or None."""
        g = self.exposure_gains
        if g is None:
            return None
        if self._camera_weight_list() is None:
            raise ValueError("exposure gains compensate the camera-weighted and multi-band blends: set camera_weights "
                             "or blend_bands > 0 too")
        if not isinstance(g, dict):
            raise ValueError("exposure_gains must be None or a dict {label: gain}, got %r" % (type(g),))
        by_label = {str(k): v for k, v in g.items()}
        labels = [str(l) for l in self.img_labels]
        unknown = sorted(set(by_label) - set(labels))
        if unknown:
            raise ValueError("exposure_gains names unknown cameras %r (cameras: %r)" % (unknown, labels))
        out = []
        for label in labels:
            v = by_label.get(label, 1.0)
            if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.integer, np.floating)) or \
                    not np.isfinite(float(v)) or float(v) < 0:
                raise ValueError("exposure_gains[%r] must be a finite gain >= 0, got %r" % (label, v))
            out.append(float(v))
        return tuple(out)

    def _graphcut_seams(self):
        """``graphcut_seams`` checked: None, or ``(digest, frames)`` only with ``blend_bands`` > 0 and without
        ``voronoi_seams``."""
        g = self.graphcut_seams
        if g is None:
            return None
        if not self._blend_bands():
            raise ValueError("graph-cut seams cut the masks of the multi-band blend: set blend_bands > 0 too")
        if self._voronoi_seams():
            raise ValueError("graph-cut seams and voronoi_seams exclude each other: set voronoi_seams = False or "
                             "call find_graphcut_seams(None)")
        if not (isinstance(g, tuple) and len(g) == 2 and isinstance(g[0], str) and len(g[1]) == len(self.img_labels)):
            raise ValueError("graphcut_seams is set by find_graphcut_seams, got %r" % (type(g),))
        return g

    def _camera_weight_list(self):
        """``camera_weights`` checked and as a list in camera order, or None when the mode is off (with
        ``blend_bands`` > 0 and no ``camera_weights``: 255 everywhere for every camera)."""
        cw = self.camera_weights
        if cw is None and self._blend_bands():
            cw = {}
        if cw is None:
            return None
        if getattr(self, "feather_log2", 0) or self.blend_weights is not None:
            raise ValueError("camera_weights / blend_bands cannot be combined with feather_log2 / blend_weights")
        by_label = {str(k): v for k, v in dict(cw).items()}
        labels = [str(l) for l in self.img_labels]
        unknown = sorted(set(by_label) - set(labels))
        if unknown:
            raise ValueError("camera_weights names unknown cameras %r (cameras: %r)" % (unknown, labels))
        out = []
        for i, label in enumerate(labels):
            m = by_label.get(label)
            if m is not None:
                m = np.asarray(m)
                # calibrated frame size: imageB of the first stage for camera 0, imageA of stage i - 1 otherwise
                st = self.stitchers[max(0, i - 1)]
                size = st.BimgSize if i == 0 else st.AimgSize
                if m.dtype != np.uint8 or m.ndim != 2 or (size is not None and m.shape != tuple(size[:2])):
                    raise ValueError("camera_weights[%r] must be a uint8 array of the camera's calibrated (h, w) %r, "
                                     "got %s %r" % (label, None if size is None else tuple(size[:2]), m.dtype, m.shape))
            out.append(m)
        return out

    # -- persistence -----------------------------------------------------------
    def save_stitcher(self, save_path):
        """Pickle the whole object (reference :138-152)."""
        try:
            with open(save_path, "wb") as output:
                for st in self.stitchers:
                    st.params_to_list()
                try:
                    pickle.dump(self, output, pickle.HIGHEST_PROTOCOL)
                finally:
                    for st in self.stitchers:
                        st.params_to_array()
            self.debugger(DEBUG_LEVEL_0, "[STITCHER]: Stitcher configuration saved")
        except IOError as e:
            self.debugger(DEBUG_LEVEL_0,
                          "[STITCHER]: Problem saving Stitcher configuration: {}".format(e), log_type="err")

    def load_stitcher(self, load_path):
        """Load a pickled configuration and RETURN the loaded object - callers
        rebind, exactly like the reference (:154-177)."""
        loaded = self
        try:
            if os.path.isfile(load_path):
                with open(load_path, "rb") as f:
                    loaded = _load_pickle(f)
                for st in loaded.stitchers:
                    st.params_to_array()
                # a Python-2 pickle read with encoding="latin1" may carry the labels as a bytes ('S') array:
                # images_dic is keyed by str
                loaded.img_labels = np.array([l.decode("latin1") if isinstance(l, bytes) else str(l)
                                              for l in loaded.img_labels])
                loaded.debugger(DEBUG_LEVEL_0, "[STITCHER]: Stitcher configuration loaded from file")
            else:
                self.debugger(DEBUG_LEVEL_0, "[STITCHER]: No Stitcher configuration file", log_type="warn")
        except IOError as e:
            self.debugger(DEBUG_LEVEL_0,
                          "[STITCHER]: Problem saving Stitcher configuration: {}".format(e), log_type="err")
        loaded._report()
        return loaded


# ---------------------------------------------------------------------------
class StitcherBase(Debugger):
    """One pair (imageB = running canvas, imageA = next camera), reference :180-529."""

    # Class-level defaults: objects unpickled from a configuration the REFERENCE saved are built without
    # __init__ and carry only the reference's fields (:190-209); re-calibrating one must still work.
    descriptor = "ORB"    # BASELINE.json config 4; "SIFT" = the reference's detector (float descriptors, L2 matching)
    nfeatures = 2000

    def __init__(self, sid=None, super_mode=False):
        self.sid = sid
        self.super_mode = super_mode
        self.reset()

    def reset(self):
        """Back to the uncalibrated state (reference :507-525)."""
        self.cachedBH = None
        self.cachedBINVH = None
        self.Bpts = None
        self.cachedAH = None
        self.cachedAINVH = None
        self.Apts = None
        self.matches = None
        self.status = None
        self.ABSize = None
        self.x_limits = None
        self.y_limits = None
        self.AimgSize = None
        self.BimgSize = None
        self.__dict__.pop("_engine", None)

    def __getstate__(self):
        state = dict(self.__dict__)
        state.pop("_engine", None)
        return state

    def __str__(self):
        return "Stitcher:{}| Matches:{}| StitcherSize:{}".format(
            self.sid, len(self.matches) if self.matches is not None else 0, self.ABSize)

    def _engine_(self):
        eng = self.__dict__.get("_engine")
        if eng is None:
            from .engine import CompositeEngine
            eng = CompositeEngine()
            self.__dict__["_engine"] = eng
        return eng

    # -- per-frame path --------------------------------------------------------
    def stitch(self, images, draw_descriptors=False):
        """Stitch ``(imageB, imageA)`` (reference :211-256)."""
        imageB, imageA = images
        if self.cachedAH is None:
            return imageB
        out = _composite(self._engine_(), [self], [imageB, imageA], batched=False, debugger=self)
        if draw_descriptors and not _is_tensor(out):
            out = self.draw_descriptors(img_src=out)
        return out

    def result_shape(self):
        """``ndarray.shape`` of what :meth:`stitch` returns once calibrated."""
        w, h = self.ABSize
        if self.super_mode:
            y0, y1, _ = slice(self.y_limits[0], self.y_limits[1]).indices(h)
            x0, x1, _ = slice(self.x_limits[0], self.x_limits[1]).indices(w)
            h, w = max(0, y1 - y0), max(0, x1 - x0)
        return (h, w) + tuple(self.AimgSize[2:])

    # -- calibration -----------------------------------------------------------
    def calibrate(self, images, ratio=0.75, reprojThresh=4.0, xoffset=10, yoffset=10):
        """Find the homography taking imageA into imageB's frame from matched
        features and derive the canvas geometry (reference :258-354)."""
        self.reset()
        imageB, imageA = images
        if _is_tensor(imageA):
            imageA = imageA.cpu().numpy()
        if _is_tensor(imageB):
            imageB = imageB.cpu().numpy()
        self.BimgSize = imageB.shape
        self.AimgSize = imageA.shape
        kpsA, featuresA = self.detectAndDescribe(imageA)
        kpsB, featuresB = self.detectAndDescribe(imageB)
        if kpsA is None or kpsB is None:
            return
        H, self.matches, self.status = self.matchKeypoints(
            kpsA=kpsA, kpsB=kpsB, featuresA=featuresA, featuresB=featuresB,
            ratio=ratio, reprojThresh=reprojThresh)
        if H is not None:
            self._geometry(H, xoffset, yoffset)
        else:
            self.reset()

    def set_homography(self, H, shapeA, shapeB, xoffset=10, yoffset=10):
        """Calibrate from a known homography (imageA -> imageB frame)."""
        matches, status = self.matches, self.status
        self.reset()
        self.matches, self.status = matches, status
        self.BimgSize = tuple(shapeB)
        self.AimgSize = tuple(shapeA)
        self._geometry(H, xoffset, yoffset)

    def _geometry(self, H, xoffset, yoffset):
        """Canvas geometry, reference :273-274 and :293-351.  Quirks kept on
        purpose: corner projections are ``int()``-truncated (Utils.py:33-35),
        the size uses ``abs(max(...))``, ROI limits split at half the canvas."""
        xoffset = abs(xoffset)
        yoffset = abs(yoffset)
        hA, wA = self.AimgSize[0], self.AimgSize[1]
        hB, wB = self.BimgSize[0], self.BimgSize[1]
        H = np.array(H, dtype=np.float64)
        cornersA = [(0, 0), (wA, 0), (wA, hA), (0, hA)]
        Apts = [get_projection_point_dst(pt_src=(p[0], p[1], 1), M=H) for p in cornersA]
        Bpts = [(0, 0), (wB, 0), (wB, hB), (0, hB)]
        both = np.concatenate((Apts, Bpts), axis=0)
        x_min = min(p[0] for p in both)
        y_min = min(p[1] for p in both)

        self.cachedBH = np.float32([[1, 0, x_min + xoffset], [0, 1, y_min + yoffset], [0, 0, 1]])
        self.cachedBINVH = np.linalg.inv(self.cachedBH)
        H[0][2] += -x_min + xoffset
        H[1][2] += -y_min + yoffset
        self.cachedAH = H
        self.cachedAINVH = np.linalg.inv(H)

        xoff = -x_min + xoffset
        yoff = -y_min + yoffset
        self.Bpts = [(xoff, yoff), (xoff + wB, yoff), (xoff + wB, hB + yoff), (xoff, hB + yoff)]
        self.Apts = [get_projection_point_dst(pt_src=(p[0], p[1], 1), M=H) for p in cornersA]
        pts = np.concatenate((self.Apts, self.Bpts), axis=0)
        xs = [p[0] for p in pts]
        ys = [p[1] for p in pts]
        self.ABSize = (int(abs(max(xs)) + xoffset), int(abs(max(ys)) + yoffset))
        self.x_limits = [max([v for v in xs if v < self.ABSize[0] * 0.5]),
                         min([v for v in xs if v > self.ABSize[0] * 0.5])]
        self.y_limits = [max([v for v in ys if v < self.ABSize[1] * 0.5]),
                         min([v for v in ys if v > self.ABSize[1] * 0.5])]

    def detectAndDescribe(self, image):
        """Key-points (float32 N x 2) and descriptors of ``image`` (reference
        :356-403).  Detection stays on the host (SURVEY.md section 8 row a6);
        ORB-2000 is BASELINE.json's recalibration workload, ``descriptor =
        "SIFT"`` selects the reference's detector."""
        if self.descriptor == "SIFT":
            if not hasattr(cv2, "SIFT_create"):
                self.debugger(DEBUG_LEVEL_0, "OpenCV has no SIFT implementation", log_type="err")
                return None, None
            det = cv2.SIFT_create()
        else:
            det = cv2.ORB_create(nfeatures=self.nfeatures)
        kps, features = det.detectAndCompute(image, None)
        if features is None:
            return None, None
        kps = np.float32([kp.pt for kp in kps]).reshape(-1, 2)
        return kps, features

    def matchKeypoints(self, kpsA, kpsB, featuresA, featuresB, ratio=0.75, reprojThresh=4.0):
        """2-NN matching + Lowe ratio test + RANSAC homography (reference
        :405-448).  Returns ``(H, matches, status)`` with ``matches`` a list of
        ``(trainIdx, queryIdx)``."""
        from . import recalib
        return recalib.match_keypoints(kpsA, kpsB, featuresA, featuresB, ratio, reprojThresh)

    def draw_descriptors(self, img_src):
        """Debug overlay of corners / ROI limits, drawn exactly like the reference's (:450-483, text through
        Calibration_Utils.print_list_text)."""
        return self._draw_descriptors_at(img_src)

    def _draw_descriptors_at(self, img_src, offset=(0, 0), canvas_size=None):
        """The overlay of a stage whose canvas origin sits at ``offset`` inside ``img_src`` and whose canvas is
        ``canvas_size = (w, h)`` - how ``Stitcher.stitch`` puts every stage's overlay into the final panorama."""
        dx, dy = int(offset[0]), int(offset[1])
        cw, ch = (img_src.shape[1], img_src.shape[0]) if canvas_size is None else (int(canvas_size[0]), int(canvas_size[1]))
        white = (255, 255, 255)

        def shifted(pts):
            return [(int(p[0]) + dx, int(p[1]) + dy) for p in pts]

        if self.Bpts is not None:
            pts = shifted(self.Bpts)
            cv2.drawContours(image=img_src, contours=np.array([pts]), contourIdx=-1, color=white, thickness=1)
            for p in pts:
                cv2.circle(img_src, p, 2, (0, 0, 255), -1)
                cv2.circle(img_src, p, 5, (0, 255, 255), 1)
        if self.Apts is not None:
            pts = shifted(self.Apts)
            cv2.drawContours(image=img_src, contours=np.array([pts]), contourIdx=-1, color=white, thickness=1)
            for p in pts:
                cv2.circle(img_src, p, 2, (0, 0, 255), -1)
                cv2.circle(img_src, p, 3, (255, 255, 0), 1)
        if self.x_limits is not None:
            for v in self.x_limits:
                cv2.line(img=img_src, pt1=(int(v) + dx, dy), pt2=(int(v) + dx, ch + dy), color=(0, 255, 0), thickness=1)
        if self.y_limits is not None:
            for v in self.y_limits:
                cv2.line(img=img_src, pt1=(dx, int(v) + dy), pt2=(cw + dx, int(v) + dy), color=(255, 255, 0), thickness=1)
        # print_list_text(str_list=[sid], origin=(20, 20), color=(0, 255, 255), thickness=1, fontScale=0.60):
        # a black outline under the coloured text (Utils.py:271-307)
        for colour, thick in (((0, 0, 0), 4), ((0, 255, 255), 1)):
            cv2.putText(img=img_src, text="{}".format(self.sid), org=(20 + dx, 20 + dy),
                        fontFace=cv2.FONT_HERSHEY_SIMPLEX, fontScale=0.60, color=colour, thickness=thick,
                        lineType=cv2.LINE_AA, bottomLeftOrigin=False)
        return img_src

    # -- persistence helpers -----------------------------------------------------
    _MATRICES = ("cachedBH", "cachedBINVH", "cachedAH", "cachedAINVH")

    def params_to_list(self):
        """Matrices -> lists of rows before pickling (reference :485-494)."""
        for name in self._MATRICES:
            if getattr(self, name) is not None:
                setattr(self, name, list(getattr(self, name)))

    def params_to_array(self):
        """Lists of rows -> arrays after loading (reference :496-505)."""
        for name in self._MATRICES:
            if getattr(self, name) is not None:
                setattr(self, name, np.asarray(getattr(self, name)))


# ---------------------------------------------------------------------------
def _segments(stages, frame_shapes, debugger=None):
    """Where the reference's shape fix-up (StitcherClass.py:226-233) strikes in this chain.

    The reference checks, at every calibrated stage, imageB (the running canvas) against
    ``BimgSize`` and imageA (the next camera) against ``AimgSize`` and resizes on any difference.
    A camera frame - or the first image while it is still the raw camera 0 - can be resized
    before the fused pass; a *composited* canvas of the wrong size cannot, so the chain is cut
    there: the stages so far run as one plan, the canvas is resized, and the remaining stages run
    as a second plan over it.  Returns a list of segments ``{a, b, base_hw, resize}``: stages
    ``[a, b)``, the height / width the segment's first image is resized to (or None), and
    ``{camera index: (h, w)}`` of the camera frames to resize."""
    tail = tuple(frame_shapes[0][2:])
    segs = []
    cur = {"a": 0, "base_hw": None, "resize": {}, "n": 0}
    cur_shape = tuple(frame_shapes[0])
    for s, st in enumerate(stages):
        if st.cachedAH is None:
            continue
        if cur_shape != tuple(st.BimgSize):
            if debugger is not None:
                debugger.debugger(DEBUG_LEVEL_0, "[STITCHER][{}] ImageB size should be {}, Image will be resized".format(
                    st.sid, st.BimgSize), log_type="warn")
            B = (int(st.BimgSize[0]), int(st.BimgSize[1]))
            if cur_shape[:2] != B:
                if cur["n"] == 0:
                    cur["base_hw"] = B
                else:
                    cur["b"] = s
                    segs.append(cur)
                    cur = {"a": s, "base_hw": B, "resize": {}, "n": 0}
        shapeA = tuple(frame_shapes[s + 1])
        if shapeA != tuple(st.AimgSize):
            if debugger is not None:
                debugger.debugger(DEBUG_LEVEL_0, "[STITCHER][{}] ImageA size should be {}, Image will be resized".format(
                    st.sid, st.AimgSize), log_type="warn")
            A = (int(st.AimgSize[0]), int(st.AimgSize[1]))
            if shapeA[:2] != A:
                cur["resize"][s + 1] = A
        cur["n"] += 1
        cur_shape = tuple(st.result_shape()[:2]) + tail
    cur["b"] = len(stages)
    segs.append(cur)
    return segs


def edge_ramp(shape, width=64):
    """A camera's edge ramp as a uint8 weight map for ``Stitcher.camera_weights``: ``min(255, (1 + distance to
    the nearest frame edge) * 255 // width)`` over a frame of ``shape`` ((h, w) or an image shape).  With it on
    every camera, overlaps blend like OpenCV's FeatherBlender."""
    h, w = int(shape[0]), int(shape[1])
    width = int(width)
    if width < 1:
        raise ValueError("ramp width must be at least 1, got %d" % width)
    yy, xx = np.mgrid[0:h, 0:w]
    d = np.minimum(np.minimum(xx, w - 1 - xx), np.minimum(yy, h - 1 - yy))
    return np.minimum(255, (1 + d) * 255 // width).astype(np.uint8)


def _composite(engine, stages, frames, batched, out=None, debugger=None, feather_log2=0, blend_weights=None,
               camera_weights=None, blend_bands=0, voronoi_seams=False, graphcut_seams=None, exposure_gains=None):
    """Run the fused kernel for this chain on these frames.  ``camera_weights``: one entry per camera (None or
    a uint8 map) for the camera-weighted blend, or None; ``blend_bands`` > 0 blends them in that many bands, with
    their masks cut at Voronoi seams when ``voronoi_seams`` or at the graph-cut seams of the frame-set
    ``graphcut_seams = (digest, frames)``; ``exposure_gains``: None or a gain per camera."""
    import torch  # local: keeps `import StitcherClass` cheap for calibration-only users

    on_device = _is_tensor(frames[0]) and frames[0].is_cuda
    shapes = [_shape_of(f)[1:] if batched else _shape_of(f) for f in frames]
    if all(st.cachedAH is None for st in stages):
        return frames[0]  # nothing calibrated: imageB passes through (reference :255-256)
    if batched and not on_device:
        raise TypeError("stitch_batch expects uint8 CUDA tensors")
    segs = _segments(stages, shapes, debugger)
    device = frames[0].device if on_device else engine.device
    n = int(frames[0].shape[0]) if batched else None

    if blend_weights is not None and len(blend_weights) != len(stages):
        raise ValueError("blend_weights must list one entry per stage (%d), got %d" % (len(stages), len(blend_weights)))
    weight_of = {} if blend_weights is None else {id(st): w for st, w in zip(stages, blend_weights)}

    def plan_for(sub_stages, sub_shapes):
        try:
            if camera_weights is not None and len(segs) > 1:
                raise PlanUnsupported("camera weights need the whole chain in one plan, but a composited canvas is "
                                      "resized at stage %d" % segs[1]["a"])
            return engine.plan_for(sub_stages, sub_shapes, device, feather_log2=feather_log2,
                                   blend_weights=[weight_of.get(id(st)) for st in sub_stages] if weight_of else None,
                                   camera_weights=camera_weights, blend_bands=blend_bands, voronoi_seams=voronoi_seams,
                                   graphcut_seams=graphcut_seams, exposure_gains=exposure_gains)
        except PlanUnsupported as e:
            if debugger is not None:
                debugger.debugger(DEBUG_LEVEL_0, "[STITCHER] {}".format(e), log_type="err")
            raise

    with torch.cuda.device(device):
        if len(segs) == 1 and segs[0]["base_hw"] is None and not segs[0]["resize"]:
            # the regular case: every frame has its calibrated size, one launch
            plan = plan_for(stages, shapes)
            if on_device:
                return plan.run(frames, out=out, n_frames=n)
            dev = [None] * len(frames)
            bands = plan.upload_bands()   # feather mode without the fused band form reports whole frames
            # only what the panorama can see of each camera crosses PCIe
            for cam, t in engine.upload_frames([l.cam for l in plan.flat.layers], frames, device, bands).items():
                dev[cam] = t
            res = plan.run(dev)
        else:
            res = None
            for i, seg in enumerate(segs):
                a, b = seg["a"], seg["b"]
                cams = [0 if res is None else None] + list(range(a + 1, b + 1))
                sub = [res if c is None else (frames[c] if on_device else engine.upload(c, frames[c], device))
                       for c in cams]
                if seg["base_hw"] is not None:
                    sub[0] = engine.resize(sub[0], seg["base_hw"], batched)
                for c, hw in seg["resize"].items():
                    sub[c - a] = engine.resize(sub[c - a], hw, batched)
                sub_shapes = [_shape_of(t)[1:] if batched else _shape_of(t) for t in sub]
                plan = plan_for(stages[a:b], sub_shapes)
                if plan is None:
                    res = sub[0]
                else:
                    res = plan.run(sub, out=out if i == len(segs) - 1 else None, n_frames=n)
            if on_device:
                return res
        return engine.download(res)   # blocking D2H into an array of its own, like cv2 allocating its result


class _CompatUnpickler(pickle.Unpickler):
    """Resolve classes pickled by the reference (module ``StitcherClass``,
    possibly under Python 2) to this module's classes."""

    def find_class(self, module, name):
        if name == "Stitcher":
            return Stitcher
        if name == "StitcherBase":
            return StitcherBase
        if module.startswith("extended_rospylogs") and name == "Debugger":
            return Debugger
        return super().find_class(module, name)


def _load_pickle(f):
    data = f.read()
    try:
        return _CompatUnpickler(_BytesReader(data)).load()
    except (UnicodeDecodeError, TypeError):
        # Python-2 pickles carry byte strings
        return _CompatUnpickler(_BytesReader(data), encoding="latin1").load()


def _BytesReader(data):
    import io
    return io.BytesIO(data)
