// Fused warp + paste compositing kernels (sm_100a).
//
// One launch produces whole panoramas: every output pixel finds the innermost layer whose
// rectangle contains it (the reference's repeated "warp A, then paste B over it",
// StitcherClass.py:239-241 applied N-1 times by :131-136) and is either copied (camera 0)
// or resampled with OpenCV's fixed-point bilinear recipe (cv2.warpPerspective, :239).
//
// Coordinate recipe (bit-exact with OpenCV's WarpPerspectiveInvoker, SURVEY.md section 8 a1):
//   (xl, yl) = pixel in the layer's own canvas frame;  xb = xl & ~63, x1 = xl & 63
//   X0 = (Mi0*xb + Mi1*yl) + Mi2  (likewise Y0, W0)          -- float64, round-to-nearest, NO fma
//   W  = W0 + Mi6*x1 ; W = W ? 32/W : 0
//   X  = rint(clamp((X0 + Mi0*x1) * W))   Y likewise          -- 1/32-px fixed point
//   out = (sum_taps w*p + 16384) >> 15, w = 32 * {(32-ay)(32-ax), (32-ay)ax, ay(32-ax), ay*ax}
// The float64 operations use the __d*_rn intrinsics, which the compiler never contracts.
#include "mcs_device.cuh"

#include <stdlib.h>
#include <string.h>

struct LayerArgs {
    McsLayer g;
    const uint8_t* src;
    long long pitch;
    long long frame_stride;
};

struct StitchArgs {
    LayerArgs L[MCS_MAX_LAYERS];
    uint8_t* dst;
    long long dst_pitch;
    long long dst_frame_stride;
    int n_layers;
    int out_w, out_h;
    int n_frames;
};

// --------------------------------------------------------------------------------------------
// per-pixel building blocks

template <int C>
__device__ __forceinline__ void load_px(const uint8_t* __restrict__ p, int (&v)[C]) {
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = __ldg(p + c);
}

// Fixed-point bilinear sample of `src` at (X, Y) in 1/32 px.  Returns whether any tap was inside
// the source.
template <int C>
__device__ __forceinline__ bool sample_u8(const uint8_t* __restrict__ src, long long pitch, int src_w,
                                          int src_h, int X, int Y, int (&out)[C]) {
    int sx = X >> 5, sy = Y >> 5;
    // saturate_cast<short> of the integer part: anything clamped is outside any legal source anyway
    sx = max(-32768, min(32767, sx));
    sy = max(-32768, min(32767, sy));
    const int ax = X & 31, ay = Y & 31;
    const bool x0in = (unsigned)sx < (unsigned)src_w, x1in = (unsigned)(sx + 1) < (unsigned)src_w;
    const bool y0in = (unsigned)sy < (unsigned)src_h, y1in = (unsigned)(sy + 1) < (unsigned)src_h;
    int p00[C], p01[C], p10[C], p11[C];
#pragma unroll
    for (int c = 0; c < C; ++c) p00[c] = p01[c] = p10[c] = p11[c] = 0;
    const uint8_t* r0 = src + (long long)sy * pitch + (long long)sx * C;
    const uint8_t* r1 = r0 + pitch;
    if (y0in && x0in) load_px<C>(r0, p00);
    if (y0in && x1in) load_px<C>(r0 + C, p01);
    if (y1in && x0in) load_px<C>(r1, p10);
    if (y1in && x1in) load_px<C>(r1 + C, p11);
    const int w00 = (32 - ay) * (32 - ax) * 32, w01 = (32 - ay) * ax * 32;
    const int w10 = ay * (32 - ax) * 32, w11 = ay * ax * 32;
#pragma unroll
    for (int c = 0; c < C; ++c)
        out[c] = (w00 * p00[c] + w01 * p01[c] + w10 * p10[c] + w11 * p11[c] + 16384) >> 15;
    return (x0in || x1in) && (y0in || y1in);
}

__device__ __forceinline__ int find_owner(const StitchArgs& a, int x, int y) {
    for (int k = 0; k < a.n_layers; ++k) {
        const McsLayer& g = a.L[k].g;
        if (x >= g.rx0 && x < g.rx1 && y >= g.ry0 && y < g.ry1) return k;
    }
    return -1;
}

// --------------------------------------------------------------------------------------------
// Variant 1 ("gather"): one thread per output pixel, consecutive lanes on consecutive pixels, the
// frames of the launch looped INSIDE the thread, source taps fetched straight from global memory.
// Handles every layout (any pitch / alignment / homography); it is the fallback of the tiled
// variant, never of a CPU path.  Owner search and the float64 coordinate recipe run once per pixel
// and launch, not once per pixel and frame; what is left per frame is the twelve tap bytes
// (neighbouring lanes share their cache lines: a warp's 32 pixels read ~110 contiguous bytes per
// source row), the integer blend and C byte stores.  Same arithmetic as sample_u8, byte loads and
// byte stores only: any pitch, any alignment.
#define MCS_GATHER_BX 64
#define MCS_GATHER_BY 4
#define MCS_GATHER_FRAMES 16   // frames per thread (grid.z covers the rest)

// WORDS: every source base, pitch and frame stride is a multiple of 4 bytes (checked by the launcher).  A pixel
// whose four taps are inside the source, with another source row below them, then fetches its taps as aligned
// 32-bit words (two or three per source row instead of 2 * C bytes) and realigns them with funnel shifts; such
// loads never leave the rows of the frame.  Border pixels keep the byte loads.
template <int C, bool WORDS>
__global__ void __launch_bounds__(MCS_GATHER_BX * MCS_GATHER_BY)
mcs_stitch_gather_frames_kernel(const __grid_constant__ StitchArgs a) {
    const int x = blockIdx.x * MCS_GATHER_BX + threadIdx.x;
    const int y = blockIdx.y * MCS_GATHER_BY + threadIdx.y;
    if (x >= a.out_w || y >= a.out_h) return;
    const int f0 = blockIdx.z * MCS_GATHER_FRAMES;
    const int n_fr = min(MCS_GATHER_FRAMES, a.n_frames - f0);
    uint8_t* out = a.dst + (long long)f0 * a.dst_frame_stride + (long long)y * a.dst_pitch + (long long)x * C;

    const int k = find_owner(a, x, y);
    if (k < 0) {   // background
        for (int f = 0; f < n_fr; ++f, out += a.dst_frame_stride)
#pragma unroll
            for (int c = 0; c < C; ++c) out[c] = 0;
        return;
    }
    const LayerArgs& L = a.L[k];
    const int xl = x - L.g.ox, yl = y - L.g.oy;
    const uint8_t* src = L.src + (long long)f0 * L.frame_stride;
    const long long fs = L.frame_stride;
    if (L.g.kind == MCS_LAYER_COPY) {
        const uint8_t* p = src + (long long)yl * L.pitch + (long long)xl * C;
        for (int f = 0; f < n_fr; ++f, p += fs, out += a.dst_frame_stride) {
            int v[C];
            load_px<C>(p, v);
#pragma unroll
            for (int c = 0; c < C; ++c) out[c] = (uint8_t)v[c];
        }
        return;
    }
    int X, Y;
    layer_coords(L.g, xl, yl, X, Y);
    const int sx = sat16(X >> 5), sy = sat16(Y >> 5);
    const int ax = X & 31, ay = Y & 31;
    const bool x0in = (unsigned)sx < (unsigned)L.g.src_w, x1in = (unsigned)(sx + 1) < (unsigned)L.g.src_w;
    const bool y0in = (unsigned)sy < (unsigned)L.g.src_h, y1in = (unsigned)(sy + 1) < (unsigned)L.g.src_h;
    const bool t00 = y0in && x0in, t01 = y0in && x1in, t10 = y1in && x0in, t11 = y1in && x1in;
    const int w00 = (32 - ay) * (32 - ax) * 32, w01 = (32 - ay) * ax * 32;
    const int w10 = ay * (32 - ax) * 32, w11 = ay * ax * 32;
    const long long pitch = L.pitch;
    const uint8_t* r0 = src + (long long)sy * pitch + (long long)sx * C;
    if (!(t00 || t01 || t10 || t11)) {   // every tap outside the source: BORDER_CONSTANT 0
        for (int f = 0; f < n_fr; ++f, out += a.dst_frame_stride)
#pragma unroll
            for (int c = 0; c < C; ++c) out[c] = 0;
        return;
    }
    if (WORDS && t00 && t11 && sy + 2 < L.g.src_h) {
        const uint32_t phase = (uint32_t)(reinterpret_cast<uintptr_t>(r0) & 3u), sh = phase * 8u;
        const uint32_t* q0 = reinterpret_cast<const uint32_t*>(r0 - phase);   // upper tap row
        const uint32_t* q1 = q0 + (pitch >> 2);                               // lower tap row
        const bool n1 = phase + 2 * C > 4, n2 = phase + 2 * C > 8;   // which words the 2 * C tap bytes reach
        const long long fs4 = fs >> 2;
        // tap weights as 16-bit pairs for IDP.2A (32768 = 32 * 32 * 32 fits an unsigned half)
        const uint32_t wu = (uint32_t)w00 | ((uint32_t)w01 << 16), wl = (uint32_t)w10 | ((uint32_t)w11 << 16);
        for (int f = 0; f < n_fr; ++f, q0 += fs4, q1 += fs4, out += a.dst_frame_stride) {
            const uint32_t u0 = __ldg(q0), u1 = n1 ? __ldg(q0 + 1) : 0u, u2 = n2 ? __ldg(q0 + 2) : 0u;
            const uint32_t v0 = __ldg(q1), v1 = n1 ? __ldg(q1 + 1) : 0u, v2 = n2 ? __ldg(q1 + 2) : 0u;
            const uint32_t lo0 = __funnelshift_r(u0, u1, sh), hi0 = __funnelshift_r(u1, u2, sh);
            const uint32_t lo1 = __funnelshift_r(v0, v1, sh), hi1 = __funnelshift_r(v1, v2, sh);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                // bytes c and C + c of the 8-byte window (lo, hi): the two taps of channel c in this row
                const uint32_t sel = (uint32_t)c | ((uint32_t)(C + c) << 4);   // IDP.2A.LO reads bytes 0 and 1 only
                const uint32_t tu = __byte_perm(lo0, hi0, sel), tl = __byte_perm(lo1, hi1, sel);
                out[c] = (uint8_t)(__dp2a_lo(wl, tl, __dp2a_lo(wu, tu, 16384u)) >> 15);
            }
        }
        return;
    }
#pragma unroll 1
    for (int f = 0; f < n_fr; ++f, r0 += fs, out += a.dst_frame_stride) {
        int p00[C], p01[C], p10[C], p11[C];
#pragma unroll
        for (int c = 0; c < C; ++c) p00[c] = p01[c] = p10[c] = p11[c] = 0;
        if (t00) load_px<C>(r0, p00);
        if (t01) load_px<C>(r0 + C, p01);
        if (t10) load_px<C>(r0 + pitch, p10);
        if (t11) load_px<C>(r0 + pitch + C, p11);
#pragma unroll
        for (int c = 0; c < C; ++c)
            out[c] = (uint8_t)((w00 * p00[c] + w01 * p01[c] + w10 * p10[c] + w11 * p11[c] + 16384) >> 15);
    }
}

// The ownership counter behind mcs_plan_owned_pixels: per layer, the output pixels it owns and
// samples from its source (COPY layers: every one; otherwise some tap must be inside the source).
// Blocks of 32 x 16 pixels; whole warps stay alive for the warp-level merge.
__global__ void __launch_bounds__(512)
mcs_owned_pixels_kernel(const __grid_constant__ StitchArgs a, unsigned long long* __restrict__ owned) {
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 16 + threadIdx.y;
    const int k = x < a.out_w && y < a.out_h ? find_owner(a, x, y) : -1;
    int counted = -1;   // layer this pixel is counted for
    if (k >= 0) {
        const McsLayer& g = a.L[k].g;
        bool touched = true;
        if (g.kind != MCS_LAYER_COPY) {
            int X, Y;
            layer_coords(g, x - g.ox, y - g.oy, X, Y);
            touched = some_tap_inside(g, X, Y);
        }
        if (touched) counted = k;
    }
    // one atomic per (warp, layer) instead of one per pixel
    const unsigned peers = __match_any_sync(0xffffffffu, counted);
    if (counted >= 0 && (int)threadIdx.x == __ffs(peers) - 1) atomicAdd(owned + counted, (unsigned long long)__popc(peers));
}

// --------------------------------------------------------------------------------------------
// Feather blend mode (extension, SURVEY.md section 8 row f1; the reference has only the overwrite
// of StitcherClass.py:240-241).  Specification: oracle/feather_model.py.  The chain's nested
// pastes are softened over F = 2^feather_log2 pixels inside every pasted rectangle:
//   value = sample of the innermost layer m whose rectangle contains the pixel
//   for k = m+1 .. n-1:   a = min(F, 1 + distance to the nearest edge of rectangle k-1)
//       a == F -> done (rectangles are nested, the distance only grows)
//       layer k touched here -> value = (a*value + (F-a)*sample_k + F/2) >> feather_log2
// Every stage rounds to uint8 like the chain it models.  Taps straight from global memory: only
// the seam bands are evaluated this way (mcs_feather_band_kernel below).
template <int C>
__device__ __forceinline__ bool sample_layer(const LayerArgs& L, int frame, int x, int y, int (&v)[C]) {
    const int xl = x - L.g.ox, yl = y - L.g.oy;
    const uint8_t* src = L.src + (long long)frame * L.frame_stride;
    if (L.g.kind == MCS_LAYER_COPY) {
        load_px<C>(src + (long long)yl * L.pitch + (long long)xl * C, v);
        return true;
    }
    int X, Y;
    layer_coords(L.g, xl, yl, X, Y);
    return sample_u8<C>(src, L.pitch, L.g.src_w, L.g.src_h, X, Y, v);
}

// Feathered value of one output pixel (all stages of the chain).
template <int C>
__device__ __forceinline__ void feather_pixel(const StitchArgs& a, int frame, int x, int y, int feather_log2,
                                              int (&v)[C]) {
    const int F = 1 << feather_log2;
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = 0;
    const int m = find_owner(a, x, y);
    if (m < 0) return;
    sample_layer<C>(a.L[m], frame, x, y, v);
    for (int k = m + 1; k < a.n_layers; ++k) {
        const McsLayer& in = a.L[k - 1].g;   // the rectangle pasted at stage k
        const int d = min(min(x - in.px0, in.px1 - 1 - x), min(y - in.py0, in.py1 - 1 - y)) + 1;
        if (d >= F) break;
        int w[C];
        if (sample_layer<C>(a.L[k], frame, x, y, w)) {
#pragma unroll
            for (int c = 0; c < C; ++c) v[c] = (d * v[c] + (F - d) * w[c] + (F >> 1)) >> feather_log2;
        }
    }
}

// Seam bands only: the feathered result differs from the overwrite result only within F pixels
// inside the border of a pasted rectangle, so the regular (tiled) kernel composites the panorama
// and this kernel then re-evaluates the band strips (plan->d_strips, at most four per stage) and
// overwrites them.  One thread per band pixel; strips may overlap, the value does not depend on
// the strip.
template <int C>
__global__ void __launch_bounds__(256)
mcs_feather_band_kernel(const __grid_constant__ StitchArgs a, const int4* __restrict__ strips,
                        const long long* __restrict__ prefix, int n_strips, int feather_log2) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= prefix[n_strips]) return;
    int s = 0;
    while (s + 1 < n_strips && prefix[s + 1] <= i) ++s;
    const int4 r = strips[s];
    const int w = r.z - r.x;
    const int j = (int)(i - prefix[s]);
    const int y = r.y + j / w, x = r.x + j % w;
    const int frame = blockIdx.z;
    int v[C];
    feather_pixel<C>(a, frame, x, y, feather_log2, v);
    uint8_t* out = a.dst + (long long)frame * a.dst_frame_stride + (long long)y * a.dst_pitch + (long long)x * C;
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = (uint8_t)v[c];
}

// Plan-time form of the same evaluation.  The chain a band pixel walks (owner layer, then every
// outer layer whose pasted rectangle border is closer than F and whose warp touches its source
// here) does not depend on the frame, and neither do the float64 source coordinates: one thread
// per band pixel records them once (mcs_feather_table_kernel), entry e of pixel i at
// ent[e * total + i] = {X, Y, layer, a} with a = weight of the value blended so far (F for the
// first entry).  Per launch, mcs_feather_apply_kernel gives each thread one band pixel and
// FEATHER_FPT consecutive frames: every entry is read once for those frames and its gathers are
// independent across them.
#define FEATHER_FPT 8

__device__ __forceinline__ void band_pixel(const int4* __restrict__ strips, const long long* __restrict__ prefix,
                                           int n_strips, long long i, int& x, int& y) {
    int s = 0;
    while (s + 1 < n_strips && prefix[s + 1] <= i) ++s;
    const int4 r = strips[s];
    const int w = r.z - r.x;
    const int j = (int)(i - prefix[s]);
    y = r.y + j / w;
    x = r.x + j % w;
}

__global__ void __launch_bounds__(256)
mcs_feather_table_kernel(const __grid_constant__ StitchArgs a, const int4* __restrict__ strips,
                         const long long* __restrict__ prefix, int n_strips, int feather_log2,
                         int2* __restrict__ band_xy, unsigned char* __restrict__ band_cnt,
                         int4* __restrict__ band_ent) {
    const long long total = prefix[n_strips];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int x, y;
    band_pixel(strips, prefix, n_strips, i, x, y);
    const int F = 1 << feather_log2;
    band_xy[i] = make_int2(x, y);
    int n = 0;
    const int m = find_owner(a, x, y);
    if (m >= 0) {
        for (int k = m; k < a.n_layers; ++k) {
            const McsLayer& g = a.L[k].g;
            int d = F;
            if (k > m) {
                const McsLayer& in = a.L[k - 1].g;   // the rectangle pasted at stage k
                d = min(min(x - in.px0, in.px1 - 1 - x), min(y - in.py0, in.py1 - 1 - y)) + 1;
                if (d >= F) break;
            }
            const int xl = x - g.ox, yl = y - g.oy;
            int X, Y;
            bool touched = true;
            if (g.kind == MCS_LAYER_COPY) {
                X = xl * 32;
                Y = yl * 32;
            } else {
                layer_coords(g, xl, yl, X, Y);
                touched = some_tap_inside(g, X, Y);
            }
            if (k == m || touched) band_ent[(size_t)n++ * total + i] = make_int4(X, Y, k, d);
        }
    }
    band_cnt[i] = (unsigned char)n;
}

template <int C>
__global__ void __launch_bounds__(256)
mcs_feather_apply_kernel(const __grid_constant__ StitchArgs a, const int2* __restrict__ band_xy,
                         const unsigned char* __restrict__ band_cnt, const int4* __restrict__ band_ent,
                         long long total, int feather_log2) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int f0 = blockIdx.y * FEATHER_FPT;
    const int nf = min(FEATHER_FPT, a.n_frames - f0);
    const int n = band_cnt[i];
    const int2 xy = band_xy[i];
    const int F = 1 << feather_log2;
    int v[FEATHER_FPT][C];
#pragma unroll
    for (int f = 0; f < FEATHER_FPT; ++f)
#pragma unroll
        for (int c = 0; c < C; ++c) v[f][c] = 0;
    for (int e = 0; e < n; ++e) {
        const int4 ent = __ldg(band_ent + (size_t)e * total + i);
        const LayerArgs& L = a.L[ent.z];
        const uint8_t* src = L.src + (long long)f0 * L.frame_stride;
        const int d = ent.w;
#pragma unroll
        for (int f = 0; f < FEATHER_FPT; ++f) {
            if (f < nf) {
                int w[C];
                sample_u8<C>(src + (long long)f * L.frame_stride, L.pitch, L.g.src_w, L.g.src_h, ent.x, ent.y, w);
#pragma unroll
                for (int c = 0; c < C; ++c)
                    v[f][c] = e == 0 ? w[c] : (d * v[f][c] + (F - d) * w[c] + (F >> 1)) >> feather_log2;
            }
        }
    }
    uint8_t* out = a.dst + (long long)f0 * a.dst_frame_stride + (long long)xy.y * a.dst_pitch + (long long)xy.x * C;
#pragma unroll
    for (int f = 0; f < FEATHER_FPT; ++f) {
        if (f < nf) {
#pragma unroll
            for (int c = 0; c < C; ++c) out[(long long)f * a.dst_frame_stride + c] = (uint8_t)v[f][c];
        }
    }
}

// --------------------------------------------------------------------------------------------
static int fill_args(const mcs_plan* plan, StitchArgs& a, const uint8_t* const* src,
                     const int64_t* src_pitch, const int64_t* src_frame_stride, int n_frames,
                     uint8_t* dst, int64_t dst_pitch, int64_t dst_frame_stride) {
    a.n_layers = plan->n_layers;
    a.out_w = plan->out_w;
    a.out_h = plan->out_h;
    a.n_frames = n_frames;
    a.dst = dst;
    a.dst_pitch = dst_pitch;
    a.dst_frame_stride = dst_frame_stride;
    for (int k = 0; k < plan->n_layers; ++k) {
        a.L[k].g = plan->layers[k];
        a.L[k].src = src ? src[k] : nullptr;
        a.L[k].pitch = src_pitch ? src_pitch[k] : 0;
        a.L[k].frame_stride = (src_frame_stride && n_frames > 1) ? src_frame_stride[k] : 0;
    }
    return MCS_OK;
}

static cudaError_t launch_gather_frames(const mcs_plan* plan, const StitchArgs& a, cudaStream_t stream) {
    dim3 block(MCS_GATHER_BX, MCS_GATHER_BY, 1);
    dim3 grid((plan->out_w + MCS_GATHER_BX - 1) / MCS_GATHER_BX, (plan->out_h + MCS_GATHER_BY - 1) / MCS_GATHER_BY,
              (a.n_frames + MCS_GATHER_FRAMES - 1) / MCS_GATHER_FRAMES);
    bool words = getenv("MCS_GATHER_BYTES") == nullptr;   // word-aligned sources: taps fetched as 32-bit words
    for (int k = 0; k < a.n_layers; ++k)
        words = words && ((reinterpret_cast<uintptr_t>(a.L[k].src) | (uintptr_t)a.L[k].pitch | (uintptr_t)a.L[k].frame_stride) & 3u) == 0;
    switch (plan->channels * 2 + (words ? 1 : 0)) {
        case 2: mcs_stitch_gather_frames_kernel<1, false><<<grid, block, 0, stream>>>(a); break;
        case 3: mcs_stitch_gather_frames_kernel<1, true><<<grid, block, 0, stream>>>(a); break;
        case 6: mcs_stitch_gather_frames_kernel<3, false><<<grid, block, 0, stream>>>(a); break;
        case 7: mcs_stitch_gather_frames_kernel<3, true><<<grid, block, 0, stream>>>(a); break;
        case 8: mcs_stitch_gather_frames_kernel<4, false><<<grid, block, 0, stream>>>(a); break;
        default: mcs_stitch_gather_frames_kernel<4, true><<<grid, block, 0, stream>>>(a); break;
    }
    mcs_count_launch(1);
    return cudaGetLastError();
}

extern "C" int mcs_stitch_u8(const mcs_plan* plan_c, const uint8_t* const* src,
                             const int64_t* src_pitch_bytes, const int64_t* src_frame_stride,
                             int n_frames, uint8_t* dst, int64_t dst_pitch_bytes,
                             int64_t dst_frame_stride, void* cuda_stream) {
    mcs_plan* plan = const_cast<mcs_plan*>(plan_c);
    MCS_CHECK_ARG(plan != nullptr, "mcs_stitch_u8: plan is NULL");
    MCS_CHECK_ARG(src && src_pitch_bytes, "mcs_stitch_u8: NULL source table");
    MCS_CHECK_ARG(n_frames >= 0 && n_frames <= 65535, "mcs_stitch_u8: n_frames=%d outside 0..65535", n_frames);
    if (n_frames == 0 || plan->out_w == 0 || plan->out_h == 0) return MCS_OK;
    MCS_CHECK_ARG(dst != nullptr, "mcs_stitch_u8: dst is NULL");
    MCS_CHECK_ARG(dst_pitch_bytes >= (int64_t)plan->out_w * plan->channels,
                  "mcs_stitch_u8: dst pitch %lld < row bytes %lld", (long long)dst_pitch_bytes,
                  (long long)plan->out_w * plan->channels);
    MCS_CHECK_ARG(n_frames == 1 || src_frame_stride != nullptr, "mcs_stitch_u8: NULL frame strides");
    for (int k = 0; k < plan->n_layers; ++k) {
        MCS_CHECK_ARG(src[k] != nullptr, "mcs_stitch_u8: source %d is NULL", k);
        MCS_CHECK_ARG(src_pitch_bytes[k] >= (int64_t)plan->layers[k].src_w * plan->channels,
                      "mcs_stitch_u8: source %d pitch %lld < row bytes", k, (long long)src_pitch_bytes[k]);
    }
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const int force = plan->force_variant;
    if (plan->mb_on) {
        if (force != 0) {
            mcs_set_error("mcs_stitch_u8: %s variant forced but unavailable: the plan blends in bands",
                          force == 1 ? "gather" : "tiled");
            return MCS_ERR_UNSUPPORTED;
        }
        const int rc = mcs_launch_multiband(plan, src, src_pitch_bytes, src_frame_stride, n_frames, dst, dst_pitch_bytes,
                                            dst_frame_stride, stream);
        if (rc == MCS_OK) plan->last_variant = 6;
        return rc;
    }
    if (plan->cw_active) {
        if (force == 2) {
            mcs_set_error("mcs_stitch_u8: tiled variant forced but unavailable: the plan blends with camera weights");
            return MCS_ERR_UNSUPPORTED;
        }
        const int rc = mcs_launch_weighted(plan, src, src_pitch_bytes, src_frame_stride, n_frames, dst, dst_pitch_bytes,
                                           dst_frame_stride, stream);
        if (rc == MCS_OK) plan->last_variant = 5;
        return rc;
    }
    const char* blocker = mcs_tiled_blocker(plan, src, src_pitch_bytes, src_frame_stride, n_frames, dst_pitch_bytes);
    if (force == 2 && blocker) {
        mcs_set_error("mcs_stitch_u8: tiled variant forced but unavailable: %s", blocker);
        return MCS_ERR_UNSUPPORTED;
    }
    StitchArgs a;
    if (!blocker && force != 1) {
        int rc = mcs_launch_tiled(plan, src, src_pitch_bytes, src_frame_stride, n_frames, dst, dst_pitch_bytes,
                              dst_frame_stride, stream);
        if (rc != MCS_OK) return rc;
        plan->last_variant = 2;
    } else {
        fill_args(plan, a, src, src_pitch_bytes, src_frame_stride, n_frames, dst, dst_pitch_bytes,
                  dst_frame_stride);
        MCS_CHECK_CUDA(launch_gather_frames(plan, a, stream));
        plan->last_variant = 1;
    }
    if (plan->band_fused && plan->last_variant == 2) {
        plan->last_variant = 4;   // the tiled kernel blended the seam bands itself (BAND tiles)
        return MCS_OK;
    }
    if (plan->blend_custom) {
        mcs_set_error("mcs_stitch_u8: weight maps / super-mode feathering exist only in the tiled variant, which cannot "
                      "serve this call: %s", blocker ? blocker : "the gather variant was forced");
        return MCS_ERR_UNSUPPORTED;
    }
    if (plan->feather_log2 > 0 && plan->n_strips > 0) {
        // feather blend: the pass above composited with the reference's overwrite; now the seam bands
        fill_args(plan, a, src, src_pitch_bytes, src_frame_stride, n_frames, dst, dst_pitch_bytes,
                  dst_frame_stride);
        const long long total = plan->strip_pixels;
        if (plan->d_band_ent) {
            dim3 tgrid((unsigned)((total + 255) / 256), (n_frames + FEATHER_FPT - 1) / FEATHER_FPT, 1);
            switch (plan->channels) {
                case 1: mcs_feather_apply_kernel<1><<<tgrid, 256, 0, stream>>>(a, plan->d_band_xy, plan->d_band_cnt, plan->d_band_ent, total, plan->feather_log2); break;
                case 3: mcs_feather_apply_kernel<3><<<tgrid, 256, 0, stream>>>(a, plan->d_band_xy, plan->d_band_cnt, plan->d_band_ent, total, plan->feather_log2); break;
                default: mcs_feather_apply_kernel<4><<<tgrid, 256, 0, stream>>>(a, plan->d_band_xy, plan->d_band_cnt, plan->d_band_ent, total, plan->feather_log2); break;
            }
            mcs_count_launch(1);
            MCS_CHECK_CUDA(cudaGetLastError());
            plan->last_variant = 3;
            return MCS_OK;
        }
        dim3 grid((unsigned)((total + 255) / 256), 1, n_frames);
        switch (plan->channels) {
            case 1: mcs_feather_band_kernel<1><<<grid, 256, 0, stream>>>(a, plan->d_strips, plan->d_strip_prefix, plan->n_strips, plan->feather_log2); break;
            case 3: mcs_feather_band_kernel<3><<<grid, 256, 0, stream>>>(a, plan->d_strips, plan->d_strip_prefix, plan->n_strips, plan->feather_log2); break;
            default: mcs_feather_band_kernel<4><<<grid, 256, 0, stream>>>(a, plan->d_strips, plan->d_strip_prefix, plan->n_strips, plan->feather_log2); break;
        }
        mcs_count_launch(1);
        MCS_CHECK_CUDA(cudaGetLastError());
        plan->last_variant = 3;
    }
    return MCS_OK;
}

extern "C" int mcs_plan_owned_pixels(const mcs_plan* plan, int64_t* owned_host, void* cuda_stream) {
    MCS_CHECK_ARG(plan != nullptr && owned_host != nullptr, "mcs_plan_owned_pixels: NULL argument");
    if (plan->cw_active || plan->mb_on) {   // counted when the weights were set
        for (int k = 0; k < plan->n_layers; ++k) owned_host[k] = (int64_t)plan->cw_contrib[k];
        return MCS_OK;
    }
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    unsigned long long* d = nullptr;
    MCS_CHECK_CUDA(cudaMalloc(&d, sizeof(unsigned long long) * MCS_MAX_LAYERS));
    int rc = MCS_OK;
    cudaError_t e = cudaMemsetAsync(d, 0, sizeof(unsigned long long) * MCS_MAX_LAYERS, stream);
    if (e == cudaSuccess && plan->out_w > 0 && plan->out_h > 0) {
        StitchArgs a;
        fill_args(plan, a, nullptr, nullptr, nullptr, 1, nullptr, 0, 0);
        const dim3 grid((plan->out_w + 31) / 32, (plan->out_h + 15) / 16, 1);
        mcs_owned_pixels_kernel<<<grid, dim3(32, 16, 1), 0, stream>>>(a, d);
        mcs_count_launch(1);
        e = cudaGetLastError();
    }
    unsigned long long h[MCS_MAX_LAYERS];
    if (e == cudaSuccess) e = cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) {
        mcs_set_error("mcs_plan_owned_pixels: %s", cudaGetErrorString(e));
        rc = MCS_ERR_CUDA;
    } else {
        for (int k = 0; k < plan->n_layers; ++k) owned_host[k] = (int64_t)h[k];
    }
    cudaFree(d);
    return rc;
}

void mcs_feather_free_table(mcs_plan* plan) {
    if (plan->d_band_xy) cudaFree(plan->d_band_xy);
    if (plan->d_band_cnt) cudaFree(plan->d_band_cnt);
    if (plan->d_band_ent) cudaFree(plan->d_band_ent);
    plan->d_band_xy = nullptr;
    plan->d_band_cnt = nullptr;
    plan->d_band_ent = nullptr;
}

void mcs_feather_build_table(mcs_plan* plan) {
    mcs_feather_free_table(plan);
    const long long total = plan->strip_pixels;
    if (plan->feather_log2 <= 0 || plan->n_strips <= 0 || total <= 0) return;
    const size_t ent_bytes = sizeof(int4) * (size_t)plan->n_layers * (size_t)total;
    if (ent_bytes > ((size_t)2 << 30)) return;   // very wide bands: evaluate on the fly instead
    {
        const char* env = getenv("MCS_FEATHER_TABLE");   // "0": keep the on-the-fly band kernel (tests)
        if (env && env[0] == '0') return;
    }
    cudaError_t e = cudaMalloc(&plan->d_band_xy, sizeof(int2) * (size_t)total);
    if (e == cudaSuccess) e = cudaMalloc(&plan->d_band_cnt, (size_t)total);
    if (e == cudaSuccess) e = cudaMalloc(&plan->d_band_ent, ent_bytes);
    if (e == cudaSuccess) {
        StitchArgs a;
        fill_args(plan, a, nullptr, nullptr, nullptr, 1, nullptr, 0, 0);
        mcs_feather_table_kernel<<<(unsigned)((total + 255) / 256), 256>>>(
            a, plan->d_strips, plan->d_strip_prefix, plan->n_strips, plan->feather_log2, plan->d_band_xy,
            plan->d_band_cnt, plan->d_band_ent);
        mcs_count_launch(1);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        mcs_feather_free_table(plan);
    }
}
