/*
 * mcs.h - C ABI of libmcs_b200.so, the sm_100a implementation of the
 * multicamera_stitching frame-compositing hot path.
 *
 * The reference (kiwicampus/multicamera_stitching) has no FFI layer: its seam
 * is the Python class API of PostScripts/Stitcher/StitcherClass.py.  Each
 * entry point below names the reference call(s) it replaces; INTEGRATION.md
 * shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; image / descriptor / point buffers are
 *     caller-owned DEVICE memory (raw CUDA device pointers), unless a
 *     parameter is documented as "host";
 *   - every function returns MCS_OK (0) or a negative MCS_ERR_* code, never
 *     throws or aborts; mcs_last_error() gives the message for the calling
 *     thread;
 *   - work is enqueued on `cuda_stream` (a cudaStream_t, NULL = default
 *     stream) and is asynchronous with respect to the host;
 *   - the library allocates nothing the caller must free except mcs_plan;
 *   - a plan serves ONE stream at a time: mcs_stitch_u8 keeps per-launch state
 *     (the run-time work counters of the tiled kernel, scratch for padded rows,
 *     the cached TMA descriptors) in the plan, so two launches of the same plan
 *     must be ordered on one stream (or by events).  Different plans are
 *     independent;
 *   - bit-exactness with cv2.warpPerspective is guaranteed for layer canvases
 *     (stage ABSize / prewarp dsize) of at least 16 rows: OpenCV splits shorter
 *     canvases into blocks wider than the 64 columns the coordinate recipe of
 *     this library assumes (imgwarp.cpp WarpPerspectiveInvoker: bh0 = min(16,
 *     rows), bw0 = min(1024 / bh0, cols)), which can move the float64 rounding
 *     of X0 + M0*x1 by one 1/32-px bucket.
 */
#ifndef MCS_B200_H
#define MCS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCS_OK               0
#define MCS_ERR_INVALID     -1   /* bad argument                              */
#define MCS_ERR_CUDA        -2   /* a CUDA runtime / driver call failed       */
#define MCS_ERR_UNSUPPORTED -3   /* valid request outside the built envelope  */
#define MCS_ERR_NOMEM       -4

#define MCS_MAX_LAYERS      16   /* cameras per panorama                      */

/* layer kinds */
#define MCS_LAYER_COPY       0   /* verbatim paste  (camera 0 / image B)      */
#define MCS_LAYER_WARP       1   /* cv2.warpPerspective(INTER_LINEAR) resample */
#define MCS_LAYER_REMAP      2   /* cv2.remap(INTER_LINEAR) through a fixed-point map */

typedef struct mcs_plan mcs_plan;

/* ABI version of this header (bumped on any signature change). */
int mcs_abi_version(void);

/* Message of the last error raised on the calling thread ("" if none). */
const char* mcs_last_error(void);

/*
 * mcs_plan_create - flatten a calibrated stitcher chain into one compositing
 * plan on the current CUDA device.
 *
 * Replaces the per-frame state walk of Stitcher.stitch (StitcherClass.py:
 * 131-136) over StitcherBase.{cachedAH, Bpts, ABSize, AimgSize, BimgSize,
 * x_limits, y_limits} (:193-209).  Layers are ordered innermost first: the
 * value of output pixel p is taken from the FIRST layer whose rectangle
 * contains p (that is the nested "paste imageB over the warped canvas" rule of
 * StitcherClass.py:239-241 applied N-1 times); pixels in no rectangle are 0.
 *
 *   n_layers   1..MCS_MAX_LAYERS
 *   channels   1, 3 or 4 (bytes per pixel of every source and of the output)
 *   layer_kind [n]    MCS_LAYER_COPY | MCS_LAYER_WARP (MCS_LAYER_REMAP: mcs_plan_create_maps)
 *   src_hw     [n*2]  source frame (height, width) of each layer
 *   fwd_h      [n*9]  row-major float64 FORWARD homography of each WARP layer,
 *                     exactly the `M` the reference hands to
 *                     cv2.warpPerspective (cachedAH); it is inverted here with
 *                     the same closed form as cv::invert.  Ignored for COPY.
 *   origin_xy  [n*2]  position, in output coordinates, of the origin of the
 *                     layer's own canvas frame (for WARP: the frame cachedAH
 *                     maps into; for COPY: where source pixel (0,0) lands)
 *   rect_xyxy  [n*4]  half-open rectangle [x0,x1) x [y0,y1), in output
 *                     coordinates, the layer (and everything it was pasted
 *                     with) occupies
 *   out_w,out_h       output panorama size (ABSize of the last stage, after
 *                     the optional super-mode crop)
 */
int mcs_plan_create(mcs_plan** out, int n_layers, int channels,
                    const int32_t* layer_kind, const int32_t* src_hw,
                    const double* fwd_h, const int32_t* origin_xy,
                    const int32_t* rect_xyxy, int out_w, int out_h);

/*
 * mcs_plan_create_maps - mcs_plan_create with MCS_LAYER_REMAP layers: the source coordinates
 * of such a layer come from a fixed-point map pair in OpenCV's own format instead of a
 * homography, and the layer is resampled exactly like cv2.remap(src, map_xy, map_frac,
 * INTER_LINEAR) with BORDER_CONSTANT 0.
 *
 * Replaces, for the per-camera pre-warp in front of the stitcher, cv2.undistort(src,
 * cameraMatrix, distCoeffs) (video_mapping_node.py:155-158, MediaPlayer/view.py:378-381,
 * Intrinsic.py:234-235; cv::undistort is initUndistortRectifyMap(CV_16SC2) + remap, and
 * Intrinsic.py:238-240 spells that form out).  The maps are calibration outputs, computed once
 * on the host; the per-frame resampling is the kernel's.
 *
 *   map_xy    host array [n_layers] of HOST pointers; for a REMAP layer k: map_hw[2k] rows x
 *             map_hw[2k+1] columns x 2 int16 (x, y) = integer source coordinates of every pixel
 *             of the layer's own canvas frame (CV_16SC2); NULL entries for other layers
 *   map_frac  the same for the uint16 interpolation-table index ((fy << 5) | fx, CV_16UC1);
 *             a NULL entry means all zero
 *   map_hw    host int32 [n_layers*2]
 * The maps are copied; the caller may free them when the call returns.  src_hw of a REMAP layer
 * is the size of the source image, the map size that of its output.  With all three NULL this is
 * mcs_plan_create.
 */
int mcs_plan_create_maps(mcs_plan** out, int n_layers, int channels,
                         const int32_t* layer_kind, const int32_t* src_hw,
                         const double* fwd_h, const int32_t* origin_xy,
                         const int32_t* rect_xyxy, int out_w, int out_h,
                         const int16_t* const* map_xy, const uint16_t* const* map_frac,
                         const int32_t* map_hw);

int mcs_plan_destroy(mcs_plan* plan);

/*
 * mcs_plan_owned_pixels - per-layer count of output pixels whose value is
 * taken from that layer and has at least one bilinear tap inside the source
 * (for COPY layers: every pixel of the visible rectangle); with camera weights
 * (mcs_plan_set_camera_weights) the pixels the layer contributes to.  Host array
 * owned[n_layers].  This is the `owned_k` of SURVEY.md section 8(d):
 *   algorithmic bytes / panorama = out_w*out_h*C + C * sum_k owned_k.
 * Synchronous (runs a counting kernel on `cuda_stream` and waits).
 */
int mcs_plan_owned_pixels(const mcs_plan* plan, int64_t* owned_host, void* cuda_stream);

/*
 * mcs_plan_source_windows - per layer, the half-open window {x0, y0, x1, y1} of SOURCE pixels
 * that the layer's owned output pixels read (host int32 xyxy[n_layers*4]).  Source bytes outside
 * the window cannot influence the panorama - they belong to the part of the camera that the
 * reference's paste (StitcherClass.py:240-241) overwrites - so a host-facing caller needs to
 * bring only the window onto the device.  Whole frames when the windows are not known (no tile
 * table, feather mode, camera weights, multi-band blend).
 */
int mcs_plan_source_windows(const mcs_plan* plan, int32_t* xyxy);

/*
 * mcs_plan_source_spans - the same information at finer grain: for every band of `band_rows`
 * source rows of layer `layer`, the half-open column range {x0, x1} its owned output pixels read
 * (host int32 x0x1[ceil(src_h / band_rows) * 2]; x0 == x1: nothing is read from the band).  A
 * camera whose visible part is not a rectangle (a sheared seam) is covered far more tightly by a
 * few row bands than by one window.
 */
int mcs_plan_source_spans(const mcs_plan* plan, int layer, int band_rows, int32_t* x0x1);

/*
 * mcs_copy_window_u8 - copy the byte window [x_byte0, x_byte0 + width_bytes) x [y0, y0 + rows)
 * of n_frames frames between two buffers of the same frame geometry (host or device, either
 * direction; pinned host memory for an asynchronous copy), leaving everything outside the window
 * untouched.  Plumbing for the host-facing sequence path: together with
 * mcs_plan_source_windows it replaces the whole-frame upload in front of mcs_stitch_u8.
 */
int mcs_copy_window_u8(void* dst, int64_t dst_pitch_bytes, int64_t dst_frame_stride, const void* src,
                       int64_t src_pitch_bytes, int64_t src_frame_stride, int64_t x_byte0,
                       int64_t width_bytes, int y0, int rows, int n_frames, void* cuda_stream);

/*
 * mcs_upload_pageable_u8 - upload byte windows of PAGEABLE host frames (the numpy frames a caller of
 * the reference's Stitcher.stitch(images_dic) holds, StitcherClass.py:114-136) through pinned staging
 * frames the caller provides.  Window i = {x_byte0, y0, width_bytes, rows} (host int64 xywh[4 * i ..])
 * of frame src[i] (row pitch src_pitch_bytes[i]; rows contiguous) goes to the same position of the
 * device frame dst[i]; staging[i] is a pinned host frame of the device frame's geometry (row pitch
 * pitch_bytes[i]).  A persistent pool of `threads` host threads copies the windows into the staging
 * frames in pieces of about piece_bytes (<= 0: 1 MiB) and the calling thread issues the
 * host-to-device copy of every piece on cuda_stream as soon as it has landed - instead of the
 * driver staging one pageable cudaMemcpy after the other on the calling thread.  Returns when the
 * last piece has been issued: the copies may still be in flight, and the staging frames must not
 * be rewritten before cuda_stream has passed them.  Several windows may share their buffers.
 */
int mcs_upload_pageable_u8(int n_windows, void* const* dst, const void* const* src, void* const* staging,
                           const int64_t* pitch_bytes, const int64_t* src_pitch_bytes, const int64_t* xywh,
                           int64_t piece_bytes, int threads, void* cuda_stream);

/*
 * mcs_stitch_u8 - composite n_frames panoramas.
 *
 * Replaces, per frame, the whole Stitcher.stitch chain (StitcherClass.py:
 * 114-136): N-1 x { cv2.warpPerspective(imageA, cachedAH, ABSize) (:239),
 * dst[By:By+hB, Bx:Bx+wB] = imageB (:240-241), super-mode crop (:248-251) }.
 *
 *   src              host array [n_layers] of device pointers, frame 0 of
 *                    each layer's source (H x W x C uint8, rows
 *                    src_pitch_bytes[k] apart)
 *   src_pitch_bytes  host array [n_layers]
 *   src_frame_stride host array [n_layers], bytes between consecutive frames
 *                    of layer k (ignored when n_frames == 1)
 *   dst              device pointer, frame 0 of the output
 *                    (out_h x out_w x C uint8, rows dst_pitch_bytes apart)
 * Every byte of the out_h x out_w*C window of each output frame is written
 * exactly once; padding bytes between rows are left untouched.
 */
int mcs_stitch_u8(const mcs_plan* plan, const uint8_t* const* src,
                  const int64_t* src_pitch_bytes, const int64_t* src_frame_stride,
                  int n_frames, uint8_t* dst, int64_t dst_pitch_bytes,
                  int64_t dst_frame_stride, void* cuda_stream);

/*
 * mcs_plan_set_feather - blend mode of the plan.  feather_log2 = 0 (default) is the
 * reference's rectangle overwrite (StitcherClass.py:240-241).  feather_log2 = n > 0 softens
 * every paste over F = 2^n pixels inside the pasted rectangle: with a = min(F, 1 + distance to
 * the nearest rectangle edge), a pixel there becomes (a*inner + (F-a)*warped + F/2) >> n where
 * the warped camera has a tap inside its source.  Extension with no reference counterpart
 * (SURVEY.md section 8 row f1); specification in oracle/feather_model.py.
 *
 * Up to feather_log2 = 5, and when no tile blends with more than two outer cameras, the seam
 * bands are blended INSIDE the tiled kernel (BAND tiles: one staged box per camera involved,
 * blend in registers, one launch; mcs_plan_source_windows / _spans then cover what the bands
 * read).  Otherwise a second pass re-evaluates the bands and the source windows are whole frames.
 * Equivalent to mcs_plan_set_blend(plan, feather_log2, NULL, NULL, NULL).
 */
int mcs_plan_set_feather(mcs_plan* plan, int feather_log2);

/*
 * mcs_plan_set_blend - the blend mode with per-stage weight maps and explicit paste rectangles.
 *   paste_xyxy   host [n_layers][4] or NULL: rectangle of layer k, in output coordinates, as the
 *                NEXT stage pasted it (the running canvas of stage k+1, StitcherClass.py:240-241)
 *                - what the visible rectangle of mcs_plan_create was before later super-mode
 *                crops (:248-251) cut it.  Must contain the visible rectangle.  NULL keeps the
 *                rectangles given to mcs_plan_create.
 *   weight_maps  host [n_layers] pointers or NULL.  weight_maps[k], k >= 1, is the uint8 weight
 *                of the running canvas at stage k in units of 1/F over layer k-1's pasted
 *                rectangle ((py1-py0) rows of (px1-px0) values, map_pitch[k] bytes apart; values
 *                above F count as F): the pixel becomes (a*canvas + (F-a)*warped + F/2) >> n
 *                where a < F and the warped camera touches its source.  A NULL entry keeps the
 *                distance ramp of mcs_plan_set_feather.  With feather_log2 = 0 a map of {0, 1}
 *                is a mask: 0 lets the warped camera through, 1 is the reference's overwrite.
 * Weight maps and cut rectangles exist only in the fused form (see above): the call fails with
 * MCS_ERR_UNSUPPORTED (and leaves the plan in overwrite mode) when the plan cannot take it.
 */
int mcs_plan_set_blend(mcs_plan* plan, int feather_log2, const int32_t* paste_xyxy,
                       const uint8_t* const* weight_maps, const int64_t* map_pitch);

/*
 * mcs_plan_set_camera_weights - the camera-weighted blend: every camera that sees an output pixel
 * contributes, weighted by its own per-pixel weight map and normalised by the summed weights (the
 * blend of OpenCV's FeatherBlender, in integers).  For output pixel p and layer k:
 *   v_k  what the layer produces at p in overwrite mode (COPY: the source pixel; WARP / REMAP: the
 *        fixed-point bilinear sample, BORDER_CONSTANT 0)
 *   w_k  the same sample (same coordinates, taps and rounding) of the layer's weight map, i.e.
 *        cv2.warpPerspective(map, cachedAH, ABSize) placed like the camera's image
 *   the contributors are the layers whose visible rectangle contains p and whose w_k > 0, S = sum w_k;
 *   out = (sum w_k * v_k + S / 2) / S per channel (integer division), 0 where S == 0.
 * One contributor gives v_k exactly.  Unlike the overwrite, the zero background of an inner canvas
 * does not hide the outer cameras.  Extension with no reference counterpart; specification in
 * oracle/camera_weight_model.py.
 *
 *   weight_maps  host [n_layers] pointers: weight_maps[k] is a uint8 map of layer k's SOURCE frame
 *                (src_h rows of src_w values, map_pitch[k] bytes apart), one value per camera pixel,
 *                so it survives recalibration; a NULL entry means 255 everywhere.
 *                weight_maps == NULL switches the mode off (the plan is the overwrite again).
 *   map_pitch    host [n_layers]
 * The maps are copied; a counting kernel then records what each layer contributes (reported by
 * mcs_plan_owned_pixels: algorithmic bytes = out_w*out_h*C + C * sum_k contributions_k) and the most
 * contributors any pixel has.  More than 4 fails with MCS_ERR_UNSUPPORTED and leaves the plan in
 * overwrite mode.  The mode excludes the stage-wise blend of mcs_plan_set_blend: setting either while
 * the other is on fails with MCS_ERR_INVALID.  mcs_stitch_u8 runs a kernel of its own for it (variant
 * 5; forcing the tiled variant fails with MCS_ERR_UNSUPPORTED), and mcs_plan_source_windows / _spans
 * report whole frames.  Synchronous.
 */
int mcs_plan_set_camera_weights(mcs_plan* plan, const uint8_t* const* weight_maps, const int64_t* map_pitch);

/*
 * mcs_plan_set_multiband - the multi-band blend of the camera-weighted panorama: OpenCV's
 * cv::detail::MultiBandBlender(try_gpu = 0, num_bands, CV_16S), bit for bit.  Every layer k with a
 * non-empty visible rectangle feeds v_k (as int16) with the mask w_k (both as defined for
 * mcs_plan_set_camera_weights) at the rectangle's corner, innermost first, into a blender prepared
 * for (0, 0, out_w, out_h); the output is the blended int16 image saturated to u8, 0 where the mask
 * of blend() is 0.  Low frequencies mix over a wide region and fine detail over a narrow one, which
 * hides seams between cameras of different exposure.  Specification in oracle/multiband_model.py.
 *
 * The plan must hold camera weights (mcs_plan_set_camera_weights; a rig that call refused only
 * because more than 4 cameras meet at a pixel counts: this mode has no contributor limit), else
 * MCS_ERR_INVALID.  num_bands = 0 goes back to the camera-weighted blend (the overwrite for such a
 * refused rig); 1..8 switch the mode on; anything else fails with MCS_ERR_INVALID.  The effective
 * count is clamped as MultiBandBlender::prepare does, to ceil(log2(max(out_w, out_h))), and
 * mcs_plan_multiband_bands reads it back (0 while the mode is off).  mcs_plan_set_camera_weights, and
 * clearing the weights, switch the mode off; the stage-wise blend of mcs_plan_set_blend excludes it.
 *
 * The weight pyramids are built here, once, on the device.  The plan also keeps a workspace for the
 * per-frame camera and panorama pyramids of MCS_MB_FRAMES frame-sets - 2 bytes * C * (sum over
 * cameras and levels of the feed regions' pixels + sum over levels >= 1 of the padded panorama's
 * pixels) per frame-set - and mcs_stitch_u8 runs the frames in sub-batches of that size, 2n + 2
 * launches each for n effective bands.  mcs_stitch_u8 reports variant 6; forcing the gather or tiled
 * variant fails with MCS_ERR_UNSUPPORTED; mcs_plan_source_windows / _spans report whole frames.
 * Synchronous.
 */
#define MCS_MB_FRAMES 16
int mcs_plan_set_multiband(mcs_plan* plan, int num_bands);
int mcs_plan_multiband_bands(const mcs_plan* plan);

/* Which kernel variant the last mcs_stitch_u8 on this plan launched
 * (diagnostics for tests / bench): 0 = none yet, 1 = gather, 2 = tiled, 3 = overwrite pass +
 * feather band pass, 4 = tiled with the seam bands blended in the same launch, 5 = camera-weighted
 * blend (mcs_plan_set_camera_weights), 6 = multi-band blend (mcs_plan_set_multiband). */
int mcs_plan_last_variant(const mcs_plan* plan);

/* Pin the kernel variant of a plan: 0 = automatic (tiled when the plan and the buffers allow
 * it, else gather), 1 = gather, 2 = tiled (mcs_stitch_u8 then fails with MCS_ERR_UNSUPPORTED
 * instead of switching).  For tests and benchmarks. */
int mcs_plan_force_variant(mcs_plan* plan, int variant);

/*
 * Source rows that are not a multiple of 4 bytes (e.g. 854 BGR pixels): the tiled variant addresses
 * rows as 4-byte words and can serve them only if every source row passed to mcs_stitch_u8 is
 * followed, inside its pitch, by ZERO bytes up to the next multiple of 4 (they stand in for the
 * BORDER_CONSTANT 0 taps right of the image).  mcs_plan_rows_need_padding tells whether the plan has
 * such a layer; mcs_plan_promise_padded_rows records the caller's promise (without it those plans
 * run the gather variant).
 */
int mcs_plan_rows_need_padding(const mcs_plan* plan);
int mcs_plan_promise_padded_rows(mcs_plan* plan, int promised);

/* "" when the tiled (TMA-staged) variant is available for this plan, else the reason it is
 * not (the gather variant then serves every call). */
const char* mcs_plan_tiled_status(const mcs_plan* plan);

/* Resident CTAs per SM of the tiled kernel as launched for this plan (0 before its first
 * tiled launch); the persistent grid is this times the SM count.  Diagnostics. */
int mcs_plan_tiled_ctas_per_sm(const mcs_plan* plan);

/* Shape of the tiled variant's work table (diagnostics; host int32 out[12]): tiles in total, FAST
 * (four-pixel group descriptors), WARP (per-pixel descriptors), COPY and ZERO tiles, general
 * passes per FAST tile, bytes of one staged source box, frames per sweep of the table, BAND tiles
 * (feather mode: tiles that blend with outer layers), 1 when the seam bands are blended inside the
 * tiled kernel (no second pass); the rest 0. */
int mcs_plan_tiled_stats(const mcs_plan* plan, int32_t* out);

/*
 * mcs_resize_linear_u8 - cv2.resize(img, (dst_w, dst_h), interpolation=cv2.INTER_LINEAR) for
 * n_frames uint8 images, bit-exact with OpenCV's 8-bit linear resize (11-bit coefficients,
 * separable with the intermediate row rounding; exact 2 x 2 decimation takes OpenCV's area
 * kernel, equal sizes copy).
 *
 * Replaces the shape fix-up of StitcherBase.stitch (StitcherClass.py:226-233: a frame whose
 * shape differs from the calibrated BimgSize / AimgSize is resized before the warp; the
 * MediaPlayer always takes this branch, MediaPlayer/view.py:408-409).
 *
 *   src, dst          device pointers to frame 0 (H x W x channels uint8, rows *_pitch_bytes
 *                     apart, frames *_frame_stride bytes apart; strides ignored when n_frames == 1)
 *   channels          1, 3 or 4
 */
int mcs_resize_linear_u8(const uint8_t* src, int src_w, int src_h, int64_t src_pitch_bytes,
                         int64_t src_frame_stride, uint8_t* dst, int dst_w, int dst_h,
                         int64_t dst_pitch_bytes, int64_t dst_frame_stride, int channels,
                         int n_frames, void* cuda_stream);

/* Number of kernels this library has launched in the calling process. */
int64_t mcs_launch_count(void);

/*
 * mcs_match_hamming_top2 - brute-force 2-nearest-neighbour Hamming matching
 * plus Lowe's ratio test, for `batch` independent image pairs.
 *
 * Replaces matcher.knnMatch(featuresA, featuresB, 2) and the ratio loop of
 * StitcherBase.matchKeypoints (StitcherClass.py:423-433) for binary (ORB)
 * descriptors.
 *
 *   q, t        device, [batch][nq_max|nt_max][desc_bytes] uint8 descriptors
 *               (query = featuresA, train = featuresB); desc_bytes % 4 == 0
 *   nq, nt      device int32[batch] actual counts per pair, or NULL (= max)
 *   ratio       keep[i] = dist0 < dist1 * ratio (evaluated in float64 like the
 *               reference's Python expression), needs both neighbours
 *   idx2,dist2  device int32 [batch][nq_max][2]: train indices / distances of
 *               the best and second best match, ties broken toward the lower
 *               train index (cv2 BFMatcher order); -1 where absent
 *   keep        device uint8 [batch][nq_max]
 */
int mcs_match_hamming_top2(const uint8_t* q, const int32_t* nq, int nq_max,
                           const uint8_t* t, const int32_t* nt, int nt_max,
                           int desc_bytes, double ratio,
                           int32_t* idx2, int32_t* dist2, uint8_t* keep,
                           int batch, void* cuda_stream);

/*
 * mcs_match_l2_top2 - the same for float32 descriptors and the L2 norm: the reference's own matcher
 * branch (SIFT descriptors, 128 floats, cv2.DescriptorMatcher_create("BruteForce") = NORM_L2,
 * StitcherClass.py:380-386 and :423-433).
 *
 *   q, t        device, [batch][nq_max|nt_max][dim] float32 descriptors, dim <= 256
 *   dist2       device float32 [batch][nq_max][2]: sqrtf of the float32 sum of squared differences,
 *               as cv2.BFMatcher(NORM_L2) reports it (bit-identical for integer-valued descriptors
 *               such as OpenCV's SIFT, whose sums are exact in float32); -1 where absent
 * Everything else as mcs_match_hamming_top2.
 */
int mcs_match_l2_top2(const float* q, const int32_t* nq, int nq_max,
                      const float* t, const int32_t* nt, int nt_max,
                      int dim, double ratio,
                      int32_t* idx2, float* dist2, uint8_t* keep,
                      int batch, void* cuda_stream);

/*
 * mcs_ransac_homography - score `k` 4-point homography hypotheses per pair,
 * one warp per hypothesis.
 *
 * Replaces the hypothesis loop inside cv2.findHomography(ptsA, ptsB, RANSAC,
 * reprojThresh) (StitcherClass.py:443-444).
 *
 *   ptsA, ptsB   device float32 [batch][n_max][2] matched points (A -> B)
 *   n            device int32[batch] point counts, or NULL (= n_max)
 *   samples      device int32 [batch][k][4] point indices of each minimal
 *                sample (host-seeded)
 *   reproj_thresh  inlier iff squared reprojection error <= thresh^2
 *   inlier_counts  device int32 [batch][k]  (-1 for a degenerate sample)
 *   H_k            device float64 [batch][k][9] hypothesis homographies
 *   best_idx       device int32 [batch]: argmax of inlier_counts (lowest
 *                  index on ties), -1 if every sample was degenerate
 *   best_mask      device uint8 [batch][n_max] inlier mask of the winner
 */
int mcs_ransac_homography(const float* ptsA, const float* ptsB, const int32_t* n,
                          int n_max, const int32_t* samples, int k,
                          float reproj_thresh, int32_t* inlier_counts,
                          double* H_k, int32_t* best_idx, uint8_t* best_mask,
                          int batch, void* cuda_stream);

/*
 * mcs_refit_homography - the host end of cv2.findHomography(ptsA, ptsB, RANSAC, reprojThresh)
 * (StitcherClass.py:443-444): least-squares refit of the winning hypothesis on its inliers
 * (normalised DLT) followed by lm_iters Levenberg-Marquardt iterations on the reprojection error
 * (OpenCV: 10).  Plain host code, no device, no stream.
 *
 *   pts_a, pts_b   host float32 [n][2] matched points (A -> B)
 *   inlier_mask    host uint8 [n] (non-zero = inlier) or NULL (= all points)
 *   h0             host float64 [9]: the winning hypothesis; returned unchanged with fewer than 4
 *                  inliers, used as the starting point with exactly 4 or when the DLT degenerates
 *   h_out          host float64 [9], h_out[8] == 1 after a refit
 */
int mcs_refit_homography(const float* pts_a, const float* pts_b, const uint8_t* inlier_mask, int n,
                         const double* h0, int lm_iters, double* h_out);

#ifdef __cplusplus
}
#endif
#endif /* MCS_B200_H */
