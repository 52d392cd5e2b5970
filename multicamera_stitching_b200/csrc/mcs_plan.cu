// Plan construction: host-side flattening checks, homography inversion, error plumbing.
#include "mcs_common.h"

#include <atomic>
#include <new>
#include <limits.h>
#include <string.h>
#include <vector>

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void mcs_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

void mcs_count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

extern "C" const char* mcs_last_error(void) { return g_err; }
extern "C" int mcs_abi_version(void) { return MCS_ABI_VERSION; }
extern "C" int64_t mcs_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

// cv::invert for a 3x3 CV_64F matrix evaluates the determinant by cofactor expansion
// along the first row, takes d = 1/det and multiplies every cofactor by d.  Reproducing
// that association (and not, say, LAPACK's LU) matters: a 2e-13 difference in the
// inverse already flips ~1 ppm of the 1/32-px coordinate buckets (SURVEY.md section 8c).
bool mcs_invert3x3(const double* s, double* t) {
    volatile double c00 = s[4] * s[8] - s[5] * s[7];
    volatile double c01 = s[3] * s[8] - s[5] * s[6];
    volatile double c02 = s[3] * s[7] - s[4] * s[6];
    volatile double det = s[0] * c00 - s[1] * c01 + s[2] * c02;
    if (det == 0.0) {
        for (int i = 0; i < 9; ++i) t[i] = 0.0;  // cv::invert zero-fills a singular result
        return false;
    }
    volatile double d = 1.0 / det;
    t[0] = c00 * d;
    t[1] = (s[2] * s[7] - s[1] * s[8]) * d;
    t[2] = (s[1] * s[5] - s[2] * s[4]) * d;
    t[3] = (s[5] * s[6] - s[3] * s[8]) * d;
    t[4] = (s[0] * s[8] - s[2] * s[6]) * d;
    t[5] = (s[2] * s[3] - s[0] * s[5]) * d;
    t[6] = c02 * d;
    t[7] = (s[1] * s[6] - s[0] * s[7]) * d;
    t[8] = (s[0] * s[4] - s[1] * s[3]) * d;
    return true;
}

static void free_maps(mcs_plan* p) {
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) {
        if (p->d_maps[k]) cudaFree(p->d_maps[k]);
        p->d_maps[k] = nullptr;
    }
}

// Uploads the fixed-point map of REMAP layer k in the packed form the kernels read:
// (X, Y) = (32 * map_x + fx, 32 * map_y + fy) with fx = frac & 31, fy = (frac >> 5) & 31, which is
// how cv::remap splits a CV_16SC2 + CV_16UC1 map pair (INTER_BITS = 5).
static int upload_map(mcs_plan* p, int k, const int16_t* xy, const uint16_t* frac, int rows, int cols) {
    const size_t n = (size_t)rows * cols;
    std::vector<int2> packed(n);
    for (size_t i = 0; i < n; ++i) {
        const int f = frac ? frac[i] : 0;
        packed[i] = make_int2((int)xy[2 * i] * 32 + (f & 31), (int)xy[2 * i + 1] * 32 + ((f >> 5) & 31));
    }
    MCS_CHECK_CUDA(cudaMalloc(&p->d_maps[k], sizeof(int2) * n));
    MCS_CHECK_CUDA(cudaMemcpy(p->d_maps[k], packed.data(), sizeof(int2) * n, cudaMemcpyHostToDevice));
    p->layers[k].map = p->d_maps[k];
    p->layers[k].map_w = cols;
    p->layers[k].map_h = rows;
    return MCS_OK;
}

extern "C" int mcs_plan_create(mcs_plan** out, int n_layers, int channels,
                               const int32_t* layer_kind, const int32_t* src_hw,
                               const double* fwd_h, const int32_t* origin_xy,
                               const int32_t* rect_xyxy, int out_w, int out_h) {
    return mcs_plan_create_maps(out, n_layers, channels, layer_kind, src_hw, fwd_h, origin_xy, rect_xyxy, out_w,
                                out_h, nullptr, nullptr, nullptr);
}

extern "C" int mcs_plan_create_maps(mcs_plan** out, int n_layers, int channels,
                                    const int32_t* layer_kind, const int32_t* src_hw,
                                    const double* fwd_h, const int32_t* origin_xy,
                                    const int32_t* rect_xyxy, int out_w, int out_h,
                                    const int16_t* const* map_xy, const uint16_t* const* map_frac,
                                    const int32_t* map_hw) {
    MCS_CHECK_ARG(out != nullptr, "mcs_plan_create: out is NULL");
    *out = nullptr;
    MCS_CHECK_ARG(n_layers >= 1 && n_layers <= MCS_MAX_LAYERS,
                  "mcs_plan_create: n_layers=%d outside 1..%d", n_layers, MCS_MAX_LAYERS);
    MCS_CHECK_ARG(channels == 1 || channels == 3 || channels == 4,
                  "mcs_plan_create: channels=%d (supported: 1, 3, 4)", channels);
    MCS_CHECK_ARG(layer_kind && src_hw && origin_xy && rect_xyxy,
                  "mcs_plan_create: NULL table pointer");
    MCS_CHECK_ARG(out_w >= 0 && out_h >= 0 && out_w < (1 << 24) && out_h < (1 << 24),
                  "mcs_plan_create: output size %dx%d out of range", out_w, out_h);

    mcs_plan* p = new (std::nothrow) mcs_plan;
    if (!p) {
        mcs_set_error("mcs_plan_create: out of host memory");
        return MCS_ERR_NOMEM;
    }
    memset(p, 0, sizeof(*p));
    p->n_layers = n_layers;
    p->channels = channels;
    p->out_w = out_w;
    p->out_h = out_h;
    cudaError_t e = cudaGetDevice(&p->device);
    if (e != cudaSuccess) {
        mcs_set_error("mcs_plan_create: cudaGetDevice failed: %s", cudaGetErrorString(e));
        delete p;
        return MCS_ERR_CUDA;
    }

    for (int k = 0; k < n_layers; ++k) {
        McsLayer& L = p->layers[k];
        L.kind = layer_kind[k];
        L.src_h = src_hw[2 * k];
        L.src_w = src_hw[2 * k + 1];
        L.ox = origin_xy[2 * k];
        L.oy = origin_xy[2 * k + 1];
        // clip the visible rectangle to the panorama
        int x0 = rect_xyxy[4 * k], y0 = rect_xyxy[4 * k + 1];
        int x1 = rect_xyxy[4 * k + 2], y1 = rect_xyxy[4 * k + 3];
        x0 = x0 < 0 ? 0 : x0;
        y0 = y0 < 0 ? 0 : y0;
        x1 = x1 > out_w ? out_w : x1;
        y1 = y1 > out_h ? out_h : y1;
        if (x1 < x0) x1 = x0;
        if (y1 < y0) y1 = y0;
        L.rx0 = x0; L.ry0 = y0; L.rx1 = x1; L.ry1 = y1;
        L.px0 = rect_xyxy[4 * k]; L.py0 = rect_xyxy[4 * k + 1]; L.px1 = rect_xyxy[4 * k + 2]; L.py1 = rect_xyxy[4 * k + 3];
        bool ok = (L.kind == MCS_LAYER_COPY || L.kind == MCS_LAYER_WARP || L.kind == MCS_LAYER_REMAP) && L.src_h > 0 &&
                  L.src_w > 0 && L.src_h < 32767 && L.src_w < 32767;  // cv2.remap's short-coordinate limit
        // canvas-frame coordinates (x - ox, y - oy) must be non-negative inside the rectangle:
        // the 64-column block split of the coordinate recipe is defined on x >= 0.
        ok = ok && (x1 == x0 || y1 == y0 || (x0 >= L.ox && y0 >= L.oy));
        if (ok && L.kind == MCS_LAYER_COPY) {
            // a paste never reads outside the source
            ok = (x1 == x0 || y1 == y0) ||
                 (x1 - L.ox <= L.src_w && y1 - L.oy <= L.src_h);
        }
        if (!ok) {
            mcs_set_error("mcs_plan_create: layer %d invalid (kind=%d src=%dx%d origin=(%d,%d) "
                          "rect=[%d,%d,%d,%d))", k, L.kind, L.src_w, L.src_h, L.ox, L.oy, x0, y0, x1, y1);
            free_maps(p);
            delete p;
            return MCS_ERR_INVALID;
        }
        if (L.kind == MCS_LAYER_REMAP) {
            const int rows = map_hw ? map_hw[2 * k] : 0, cols = map_hw ? map_hw[2 * k + 1] : 0;
            if (!map_xy || !map_xy[k] || rows <= 0 || cols <= 0 || rows >= (1 << 15) || cols >= (1 << 15)) {
                mcs_set_error("mcs_plan_create_maps: layer %d is a REMAP layer without a valid map (%d x %d)", k,
                              rows, cols);
                free_maps(p);
                delete p;
                return MCS_ERR_INVALID;
            }
            // the map must cover the visible rectangle (in the layer's own canvas frame)
            if (x1 > x0 && y1 > y0 && (x1 - L.ox > cols || y1 - L.oy > rows)) {
                mcs_set_error("mcs_plan_create_maps: layer %d: rectangle [%d,%d,%d,%d) exceeds its %d x %d map at "
                              "origin (%d,%d)", k, x0, y0, x1, y1, cols, rows, L.ox, L.oy);
                free_maps(p);
                delete p;
                return MCS_ERR_INVALID;
            }
            const int rc = upload_map(p, k, map_xy[k], map_frac ? map_frac[k] : nullptr, rows, cols);
            if (rc != MCS_OK) {
                free_maps(p);
                delete p;
                return rc;
            }
            L.mi[0] = L.mi[4] = L.mi[8] = 1.0;
        } else if (L.kind == MCS_LAYER_WARP) {
            if (!fwd_h) {
                mcs_set_error("mcs_plan_create: fwd_h is NULL but layer %d is a WARP layer", k);
                free_maps(p);
                delete p;
                return MCS_ERR_INVALID;
            }
            mcs_invert3x3(fwd_h + 9 * k, L.mi);  // singular -> all-zero inverse, as cv2 does
            L.affine = (L.mi[6] == 0.0 && L.mi[7] == 0.0) ? 1 : 0;
            // W is affine in the pixel position, so its extremes over the rectangle sit at the corners
            if (x1 > x0 && y1 > y0) {
                double lo = 1e300, hi = -1e300;
                for (int cx = 0; cx < 2; ++cx)
                    for (int cy = 0; cy < 2; ++cy) {
                        const double xl = (cx ? x1 - 1 : x0) - L.ox, yl = (cy ? y1 - 1 : y0) - L.oy;
                        const double W = L.mi[6] * xl + L.mi[7] * yl + L.mi[8];
                        lo = W < lo ? W : lo;
                        hi = W > hi ? W : hi;
                    }
                const bool pos = lo >= 1e-3 && hi <= 1e6, neg = hi <= -1e-3 && lo >= -1e6;
                L.w_safe = (pos || neg) ? 1 : 0;
            }
        } else {
            L.mi[0] = L.mi[4] = L.mi[8] = 1.0;
            L.affine = 1;
        }
    }
    mcs_plan_build_tiles(p);   // never fails the plan: the gather variant covers what it cannot
    *out = p;
    return MCS_OK;
}

extern "C" int mcs_plan_destroy(mcs_plan* plan) {
    if (!plan) return MCS_OK;
    mcs_feather_free_table(plan);
    if (plan->d_strips) cudaFree(plan->d_strips);
    if (plan->d_strip_prefix) cudaFree(plan->d_strip_prefix);
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) {
        if (plan->d_wmap[k]) cudaFree(plan->d_wmap[k]);
        if (plan->d_cwmap[k]) cudaFree(plan->d_cwmap[k]);
    }
    mcs_multiband_free(plan);
    mcs_plan_free_tiles(plan);
    free_maps(plan);
    delete plan;
    return MCS_OK;
}

extern "C" int mcs_plan_rows_need_padding(const mcs_plan* plan) { return plan ? plan->rows_need_pad : 0; }

extern "C" int mcs_plan_promise_padded_rows(mcs_plan* plan, int promised) {
    MCS_CHECK_ARG(plan != nullptr, "mcs_plan_promise_padded_rows: plan is NULL");
    plan->pad_promised = promised ? 1 : 0;
    plan->cache_valid = 0;
    return MCS_OK;
}

extern "C" int mcs_plan_source_windows(const mcs_plan* plan, int32_t* xyxy) {
    MCS_CHECK_ARG(plan != nullptr && xyxy != nullptr, "mcs_plan_source_windows: NULL argument");
    // The feather band samples outer cameras inside the pasted rectangles, i.e. outside the
    // pixels they own: there every frame counts in full.
    // The camera-weighted and multi-band blends sample every camera wherever its rectangle reaches:
    // whole frames too.
    const bool known = plan->src_win_valid && !plan->cw_active && !plan->mb_on &&
                       ((plan->feather_log2 == 0 && !plan->blend_custom) || plan->band_fused);
    for (int k = 0; k < plan->n_layers; ++k) {
        xyxy[4 * k + 0] = known ? plan->src_win[k][0] : 0;
        xyxy[4 * k + 1] = known ? plan->src_win[k][1] : 0;
        xyxy[4 * k + 2] = known ? plan->src_win[k][2] : plan->layers[k].src_w;
        xyxy[4 * k + 3] = known ? plan->src_win[k][3] : plan->layers[k].src_h;
    }
    return MCS_OK;
}

extern "C" int mcs_plan_source_spans(const mcs_plan* plan, int layer, int band_rows, int32_t* x0x1) {
    MCS_CHECK_ARG(plan != nullptr && x0x1 != nullptr && band_rows > 0, "mcs_plan_source_spans: bad argument");
    MCS_CHECK_ARG(layer >= 0 && layer < plan->n_layers, "mcs_plan_source_spans: layer %d outside 0..%d", layer,
                  plan->n_layers - 1);
    const McsLayer& L = plan->layers[layer];
    const int n_bands = (L.src_h + band_rows - 1) / band_rows;
    const int* span = plan->h_row_span[layer];
    const bool known = plan->src_win_valid && !plan->cw_active && !plan->mb_on &&
                       ((plan->feather_log2 == 0 && !plan->blend_custom) || plan->band_fused) && span != nullptr;
    for (int b = 0; b < n_bands; ++b) {
        int x0 = known ? INT_MAX : 0, x1 = known ? INT_MIN : L.src_w;
        for (int r = b * band_rows; known && r < (b + 1) * band_rows && r < L.src_h; ++r) {
            x0 = span[2 * r] < x0 ? span[2 * r] : x0;
            x1 = span[2 * r + 1] > x1 ? span[2 * r + 1] : x1;
        }
        if (x1 <= x0) x0 = x1 = 0;
        x0x1[2 * b] = x0 < 0 ? 0 : x0;
        x0x1[2 * b + 1] = x1 > L.src_w ? L.src_w : x1;
    }
    return MCS_OK;
}

// Strided frame-window copy in either direction (one cudaMemcpy3DAsync: width x rows x frames).
extern "C" int mcs_copy_window_u8(void* dst, int64_t dst_pitch_bytes, int64_t dst_frame_stride, const void* src,
                                  int64_t src_pitch_bytes, int64_t src_frame_stride, int64_t x_byte0,
                                  int64_t width_bytes, int y0, int rows, int n_frames, void* cuda_stream) {
    MCS_CHECK_ARG(dst != nullptr && src != nullptr, "mcs_copy_window_u8: NULL buffer");
    MCS_CHECK_ARG(x_byte0 >= 0 && width_bytes >= 0 && y0 >= 0 && rows >= 0 && n_frames >= 0,
                  "mcs_copy_window_u8: negative extent");
    if (width_bytes == 0 || rows == 0 || n_frames == 0) return MCS_OK;
    MCS_CHECK_ARG(x_byte0 + width_bytes <= dst_pitch_bytes && x_byte0 + width_bytes <= src_pitch_bytes,
                  "mcs_copy_window_u8: window wider than a row");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const bool as3d = n_frames == 1 || (dst_frame_stride % dst_pitch_bytes == 0 && src_frame_stride % src_pitch_bytes == 0);
    if (as3d) {
        cudaMemcpy3DParms p;
        memset(&p, 0, sizeof(p));
        const size_t dst_rows = n_frames == 1 ? (size_t)(y0 + rows) : (size_t)(dst_frame_stride / dst_pitch_bytes);
        const size_t src_rows = n_frames == 1 ? (size_t)(y0 + rows) : (size_t)(src_frame_stride / src_pitch_bytes);
        p.srcPtr = make_cudaPitchedPtr(const_cast<void*>(src), (size_t)src_pitch_bytes, (size_t)src_pitch_bytes, src_rows);
        p.dstPtr = make_cudaPitchedPtr(dst, (size_t)dst_pitch_bytes, (size_t)dst_pitch_bytes, dst_rows);
        p.srcPos = make_cudaPos((size_t)x_byte0, (size_t)y0, 0);
        p.dstPos = make_cudaPos((size_t)x_byte0, (size_t)y0, 0);
        p.extent = make_cudaExtent((size_t)width_bytes, (size_t)rows, (size_t)n_frames);
        p.kind = cudaMemcpyDefault;
        MCS_CHECK_CUDA(cudaMemcpy3DAsync(&p, stream));
        return MCS_OK;
    }
    for (int f = 0; f < n_frames; ++f) {
        const char* s = static_cast<const char*>(src) + (size_t)f * src_frame_stride + (size_t)y0 * src_pitch_bytes + x_byte0;
        char* d = static_cast<char*>(dst) + (size_t)f * dst_frame_stride + (size_t)y0 * dst_pitch_bytes + x_byte0;
        MCS_CHECK_CUDA(cudaMemcpy2DAsync(d, (size_t)dst_pitch_bytes, s, (size_t)src_pitch_bytes, (size_t)width_bytes,
                                         (size_t)rows, cudaMemcpyDefault, stream));
    }
    return MCS_OK;
}

extern "C" int mcs_plan_last_variant(const mcs_plan* plan) { return plan ? plan->last_variant : 0; }

extern "C" int mcs_plan_force_variant(mcs_plan* plan, int variant) {
    MCS_CHECK_ARG(plan != nullptr && variant >= 0 && variant <= 2, "mcs_plan_force_variant: bad argument");
    plan->force_variant = variant;
    return MCS_OK;
}

extern "C" const char* mcs_plan_tiled_status(const mcs_plan* plan) {
    if (!plan) return "no plan";
    return plan->tiled_ok ? "" : plan->tiled_why;
}

extern "C" int mcs_plan_tiled_ctas_per_sm(const mcs_plan* plan) { return plan ? plan->grid_ctas_per_sm : 0; }

extern "C" int mcs_plan_tiled_stats(const mcs_plan* plan, int32_t* out) {
    MCS_CHECK_ARG(plan != nullptr && out != nullptr, "mcs_plan_tiled_stats: NULL argument");
    for (int i = 0; i < 12; ++i) out[i] = 0;
    if (!plan->tiled_ok) return MCS_OK;
    out[0] = plan->n_tiles;
    for (int c = 1; c < MCS_N_CLASSES; ++c) out[c] = plan->class_first[c + 1] - plan->class_first[c];
    out[8] = plan->class_first[1] - plan->class_first[0];
    out[9] = plan->band_fused;
    out[5] = plan->fast_passes;
    out[6] = plan->box_bytes;
    out[7] = plan->frame_block;
    return MCS_OK;
}

static void free_strips(mcs_plan* plan) {
    mcs_feather_free_table(plan);
    if (plan->d_strips) cudaFree(plan->d_strips);
    if (plan->d_strip_prefix) cudaFree(plan->d_strip_prefix);
    plan->d_strips = nullptr;
    plan->d_strip_prefix = nullptr;
    plan->n_strips = 0;
    plan->strip_pixels = 0;
}

// The tile table depends on the blend mode (feather mode adds BAND tiles and their boxes).
static void rebuild_tiles(mcs_plan* plan) {
    mcs_plan_free_tiles(plan);
    plan->cache_valid = 0;        // TMA descriptors carry the box sizes
    plan->grid_ctas_per_sm = 0;   // and the kernel's shared-memory footprint changes
    mcs_plan_build_tiles(plan);
}

static void free_wmaps(mcs_plan* plan) {
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) {
        if (plan->d_wmap[k]) cudaFree(plan->d_wmap[k]);
        plan->d_wmap[k] = nullptr;
    }
}

extern "C" int mcs_plan_set_feather(mcs_plan* plan, int feather_log2) {
    return mcs_plan_set_blend(plan, feather_log2, nullptr, nullptr, nullptr);
}

extern "C" int mcs_plan_set_blend(mcs_plan* plan, int feather_log2, const int32_t* paste_xyxy,
                                  const uint8_t* const* weight_maps, const int64_t* map_pitch) {
    MCS_CHECK_ARG(plan != nullptr, "mcs_plan_set_blend: plan is NULL");
    MCS_CHECK_ARG(feather_log2 >= 0 && feather_log2 <= 12, "mcs_plan_set_blend: feather_log2=%d outside 0..12",
                  feather_log2);
    bool any_map = false;
    for (int k = 1; weight_maps && k < plan->n_layers; ++k) any_map = any_map || weight_maps[k] != nullptr;
    MCS_CHECK_ARG(!any_map || map_pitch != nullptr, "mcs_plan_set_blend: weight maps without their pitches");
    MCS_CHECK_ARG(!any_map || feather_log2 <= MCS_BAND_MAX_LOG2,
                  "mcs_plan_set_blend: weight maps take feather_log2 <= %d (got %d)", MCS_BAND_MAX_LOG2, feather_log2);
    MCS_CHECK_ARG(!(plan->cw_active || plan->mb_on) || (feather_log2 == 0 && !any_map),
                  "mcs_plan_set_blend: the plan blends with camera weights; clear them first");
    free_strips(plan);
    free_wmaps(plan);
    const bool had = plan->feather_log2 > 0 || plan->blend_custom;
    plan->feather_log2 = 0;
    plan->blend_custom = 0;
    if (paste_xyxy) {
        for (int k = 0; k < plan->n_layers; ++k) {
            McsLayer& L = plan->layers[k];
            L.px0 = paste_xyxy[4 * k]; L.py0 = paste_xyxy[4 * k + 1]; L.px1 = paste_xyxy[4 * k + 2]; L.py1 = paste_xyxy[4 * k + 3];
            const bool empty = L.rx1 <= L.rx0 || L.ry1 <= L.ry0;
            if (!empty && (L.px0 > L.rx0 || L.py0 > L.ry0 || L.px1 < L.rx1 || L.py1 < L.ry1)) {
                mcs_set_error("mcs_plan_set_blend: layer %d: the pasted rectangle [%d,%d,%d,%d) does not contain the visible "
                              "one [%d,%d,%d,%d)", k, L.px0, L.py0, L.px1, L.py1, L.rx0, L.ry0, L.rx1, L.ry1);
                return MCS_ERR_INVALID;
            }
        }
    }
    bool cut = false;   // some rectangle was cut after it was pasted (super-mode crops): distances run to the pasted edges
    for (int k = 0; k + 1 < plan->n_layers; ++k) {
        const McsLayer& L = plan->layers[k];
        if (L.rx1 > L.rx0 && L.ry1 > L.ry0)
            cut = cut || L.px0 != L.rx0 || L.py0 != L.ry0 || L.px1 != L.rx1 || L.py1 != L.ry1;
    }
    if (feather_log2 == 0 && !any_map) {
        if (had) rebuild_tiles(plan);
        return MCS_OK;
    }
    // the blend walks the nested rectangles: they must be nested
    for (int k = 1; k < plan->n_layers; ++k) {
        const McsLayer& o = plan->layers[k];
        const McsLayer& i = plan->layers[k - 1];
        const bool empty_i = i.rx1 <= i.rx0 || i.ry1 <= i.ry0;
        if (!empty_i && (o.rx0 > i.rx0 || o.ry0 > i.ry0 || o.rx1 < i.rx1 || o.ry1 < i.ry1)) {
            mcs_set_error("mcs_plan_set_blend: layer rectangles are not nested (layer %d)", k);
            return MCS_ERR_UNSUPPORTED;
        }
    }
    for (int k = 1; any_map && k < plan->n_layers; ++k) {
        if (!weight_maps[k]) continue;
        const McsLayer& in = plan->layers[k - 1];
        const int mw = in.px1 - in.px0, mh = in.py1 - in.py0;
        if (mw <= 0 || mh <= 0) continue;
        if (map_pitch[k] < mw) {
            mcs_set_error("mcs_plan_set_blend: weight map %d: pitch %lld < %d columns", k, (long long)map_pitch[k], mw);
            free_wmaps(plan);
            return MCS_ERR_INVALID;
        }
        cudaError_t e = cudaMalloc(&plan->d_wmap[k], (size_t)mw * mh);
        if (e == cudaSuccess)
            e = cudaMemcpy2D(plan->d_wmap[k], (size_t)mw, weight_maps[k], (size_t)map_pitch[k], (size_t)mw, (size_t)mh,
                             cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            free_wmaps(plan);
            mcs_set_error("mcs_plan_set_blend: weight map %d: %s", k, cudaGetErrorString(e));
            return MCS_ERR_CUDA;
        }
    }
    plan->blend_custom = (any_map || cut) ? 1 : 0;
    if (plan->blend_custom) {
        // weight maps / cut rectangles exist only in the fused form (BAND tiles of the tiled kernel)
        plan->feather_log2 = feather_log2;
        rebuild_tiles(plan);
        if (!plan->band_fused) {
            plan->feather_log2 = 0;
            plan->blend_custom = 0;
            free_wmaps(plan);
            rebuild_tiles(plan);
            mcs_set_error("mcs_plan_set_blend: weight maps and super-mode crops need the fused band form of the tiled variant "
                          "(feather_log2 <= %d, at most %d outer layers per tile, tiled variant available)",
                          MCS_BAND_MAX_LOG2, MCS_BAND_MAX_OVERLAYS);
            return MCS_ERR_UNSUPPORTED;
        }
        return MCS_OK;
    }
    // Band strips: inside the rectangle pasted at stage k (that of layer k-1), the pixels closer
    // than F - 1 to its border: top and bottom strips over the full width, left and right strips
    // over the rows between them.
    const int F = 1 << feather_log2, B = F - 1;
    int4 strips[4 * MCS_MAX_LAYERS];
    long long prefix[4 * MCS_MAX_LAYERS + 1];
    int n = 0;
    prefix[0] = 0;
    auto add = [&](int x0, int y0, int x1, int y1) {
        if (x1 > x0 && y1 > y0) {
            strips[n] = make_int4(x0, y0, x1, y1);
            prefix[n + 1] = prefix[n] + (long long)(x1 - x0) * (y1 - y0);
            ++n;
        }
    };
    for (int k = 1; k < plan->n_layers && B > 0; ++k) {
        const McsLayer& r = plan->layers[k - 1];
        if (r.rx1 <= r.rx0 || r.ry1 <= r.ry0) continue;
        const int yt = r.ry0 + B < r.ry1 ? r.ry0 + B : r.ry1;          // end of the top strip
        const int yb = r.ry1 - B > yt ? r.ry1 - B : yt;                  // start of the bottom strip
        add(r.rx0, r.ry0, r.rx1, yt);
        add(r.rx0, yb, r.rx1, r.ry1);
        const int xl = r.rx0 + B < r.rx1 ? r.rx0 + B : r.rx1;
        const int xr = r.rx1 - B > xl ? r.rx1 - B : xl;
        add(r.rx0, yt, xl, yb);
        add(xr, yt, r.rx1, yb);
    }
    if (n > 0) {
        cudaError_t e = cudaMalloc(&plan->d_strips, sizeof(int4) * n);
        if (e == cudaSuccess) e = cudaMalloc(&plan->d_strip_prefix, sizeof(long long) * (n + 1));
        if (e == cudaSuccess) e = cudaMemcpy(plan->d_strips, strips, sizeof(int4) * n, cudaMemcpyHostToDevice);
        if (e == cudaSuccess)
            e = cudaMemcpy(plan->d_strip_prefix, prefix, sizeof(long long) * (n + 1), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            free_strips(plan);
            mcs_set_error("mcs_plan_set_blend: %s", cudaGetErrorString(e));
            return MCS_ERR_CUDA;
        }
        plan->n_strips = n;
        plan->strip_pixels = prefix[n];
    }
    plan->feather_log2 = feather_log2;
    mcs_feather_build_table(plan);
    rebuild_tiles(plan);   // the tile table knows the seam bands (BAND tiles): the tiled kernel then blends them itself
    return MCS_OK;
}

static void free_cwmaps(mcs_plan* plan) {
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) {
        if (plan->d_cwmap[k]) cudaFree(plan->d_cwmap[k]);
        plan->d_cwmap[k] = nullptr;
    }
    plan->cw_active = 0;
    plan->cw_maps = 0;
    plan->mb_on = 0;
    mcs_multiband_free(plan);
}

extern "C" int mcs_plan_set_camera_weights(mcs_plan* plan, const uint8_t* const* weight_maps, const int64_t* map_pitch) {
    MCS_CHECK_ARG(plan != nullptr, "mcs_plan_set_camera_weights: plan is NULL");
    bool any_map = false;
    for (int k = 0; weight_maps && k < plan->n_layers; ++k) any_map = any_map || weight_maps[k] != nullptr;
    MCS_CHECK_ARG(!any_map || map_pitch != nullptr, "mcs_plan_set_camera_weights: weight maps without their pitches");
    for (int k = 0; any_map && k < plan->n_layers; ++k)
        MCS_CHECK_ARG(!weight_maps[k] || map_pitch[k] >= plan->layers[k].src_w,
                      "mcs_plan_set_camera_weights: weight map %d: pitch %lld < %d columns", k, (long long)map_pitch[k],
                      plan->layers[k].src_w);
    MCS_CHECK_ARG(!weight_maps || (plan->feather_log2 == 0 && !plan->blend_custom),
                  "mcs_plan_set_camera_weights: the plan feathers its pastes (mcs_plan_set_blend); switch that off first");
    free_cwmaps(plan);
    if (!weight_maps) return MCS_OK;
    for (int k = 0; k < plan->n_layers; ++k) {
        if (!weight_maps[k]) continue;
        const McsLayer& L = plan->layers[k];
        cudaError_t e = cudaMalloc(&plan->d_cwmap[k], (size_t)L.src_w * L.src_h);
        if (e == cudaSuccess)
            e = cudaMemcpy2D(plan->d_cwmap[k], (size_t)L.src_w, weight_maps[k], (size_t)map_pitch[k], (size_t)L.src_w,
                             (size_t)L.src_h, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            free_cwmaps(plan);
            mcs_set_error("mcs_plan_set_camera_weights: weight map %d: %s", k, cudaGetErrorString(e));
            return MCS_ERR_CUDA;
        }
    }
    int most = 0;
    const int rc = mcs_camera_weights_count(plan, plan->cw_contrib, &most);
    if (rc != MCS_OK) {
        free_cwmaps(plan);
        return rc;
    }
    plan->cw_maps = 1;
    if (most > MCS_CW_MAX_CONTRIB) {   // the maps stay held for mcs_plan_set_multiband
        mcs_set_error("mcs_plan_set_camera_weights: %d cameras with non-zero weight meet at one output pixel (at most %d "
                      "blend); lower the weights of some of them there", most, MCS_CW_MAX_CONTRIB);
        return MCS_ERR_UNSUPPORTED;
    }
    plan->cw_active = 1;
    return MCS_OK;
}

extern "C" int mcs_plan_set_multiband(mcs_plan* plan, int num_bands) {
    MCS_CHECK_ARG(plan != nullptr, "mcs_plan_set_multiband: plan is NULL");
    MCS_CHECK_ARG(num_bands >= 0 && num_bands <= MCS_MB_MAX_LEVELS - 1, "mcs_plan_set_multiband: num_bands=%d outside 0..%d",
                  num_bands, MCS_MB_MAX_LEVELS - 1);
    MCS_CHECK_ARG(plan->cw_maps, "mcs_plan_set_multiband: the plan has no camera weights (mcs_plan_set_camera_weights)");
    MCS_CHECK_ARG(plan->feather_log2 == 0 && !plan->blend_custom,
                  "mcs_plan_set_multiband: the plan feathers its pastes (mcs_plan_set_blend); switch that off first");
    plan->mb_on = 0;
    mcs_multiband_free(plan);
    if (num_bands == 0) return MCS_OK;
    const int rc = mcs_multiband_build(plan, num_bands);
    if (rc != MCS_OK) return rc;
    plan->mb_on = 1;
    return MCS_OK;
}

extern "C" int mcs_plan_multiband_bands(const mcs_plan* plan) { return plan && plan->mb_on ? plan->mb_bands : 0; }
