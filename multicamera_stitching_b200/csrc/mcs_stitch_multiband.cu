// Multi-band blend of the camera-weighted panorama (mcs_plan_set_multiband, sm_100a): OpenCV's
// cv::detail::MultiBandBlender with CV_16S weights, fed with every camera's overwrite sample v_k and
// weight sample w_k over its visible rectangle.  Specification: oracle/multiband_model.py.  Integer
// only, bit-exact with OpenCV's CPU code.
//
// Geometry (host, plan time): with n bands the panorama ROI is padded to multiples of 2^n; each camera
// keeps the region feed() keeps - its rectangle grown by 3 * 2^n, clipped, corners aligned to 2^n - so
// that level i of the camera's pyramids is exactly the region shifted right by i.
//
// Plan time (constants of the calibration): per camera the weight pyramid (level 0 = w + (w != 0)
// inside the rectangle, 0 in the border; pyrDown for the rest) and per level the weight sums.
//
// Per sub-batch of MCS_MB_FRAMES frame-sets, 2n + 2 launches:
//   1. mb_level0_kernel      level 0 of every camera: the sample at the BORDER_REFLECT index of the
//                            rectangle, as int16
//   2. mb_pyrdown_kernel     n launches, the Gaussian pyramids of all cameras and frames
//   3. mb_blend_kernel       n + 1 launches, level n first: per panorama pixel of level i, every
//                            covering camera's Laplacian G_i - pyrUp(G_{i+1}) times its weight >> 8,
//                            summed in int32 (= the int16 running sum of OpenCV modulo 2^16), normalised
//                            by (sum of weights + 1); plus pyrUp of the restored level i + 1 (the collapse,
//                            saturating).  Level 0 stores u8 into the caller's output, 0 where the summed
//                            weight is 0.
#include "mcs_device.cuh"

#include <math.h>
#include <string.h>

#define MB_BX 32
#define MB_BY 8

struct MbCam {
    int k;                   // layer
    int x0, y0, x1, y1;      // visible rectangle, clipped to the panorama
    int tlx, tly, bw, bh;    // feed region: origin in the padded ROI and size (multiples of 2^n)
};

struct MbArgs {
    McsLayer g[MCS_MAX_LAYERS];
    MbCam cam[MCS_MAX_LAYERS];
    long long off[MCS_MAX_LAYERS][MCS_MB_MAX_LEVELS];    // camera j, level i: offset (int16 elements) in one frame's pyramids
    long long woff[MCS_MAX_LAYERS][MCS_MB_MAX_LEVELS];   // camera j, level i: offset of its weight level
    long long poff[MCS_MB_MAX_LEVELS];                   // panorama level i >= 1: offset in one frame's pyramid
    long long soff[MCS_MB_MAX_LEVELS];                   // level i: offset of the weight sums
    long long cam_elems, pan_elems;                      // int16 elements of one frame's camera / panorama pyramids
    int n_cams, n_bands, roi_w, roi_h, out_w, out_h, channels;
    // device buffers
    const uint8_t* wmap[MCS_MAX_LAYERS];
    int16_t* wpyr;
    int16_t* wsum;
    int16_t* ws_cam;
    int16_t* ws_pan;
    // per launch
    const uint8_t* src[MCS_MAX_LAYERS];
    long long pitch[MCS_MAX_LAYERS];
    long long frame_stride[MCS_MAX_LAYERS];
    uint8_t* dst;
    long long dst_pitch, dst_frame_stride;
    // plan time: per layer the seam-cut weights over its rectangle (mcs_seams.cu), nullptr = sample the map
    const uint8_t* seam[MCS_MAX_LAYERS];
    // per launch, GAIN: per layer the 256-entry exposure table (mcs_exposure.cu)
    const uint8_t* lut;
};

struct McsMultiband {
    MbArgs a;                // geometry and buffers; the launcher fills the per-launch fields of a copy
    int max_bw, max_bh;
    size_t ws_bytes;
};

__device__ __forceinline__ int refl(int p, int n, int delta) {   // cv::borderInterpolate, REFLECT / REFLECT_101
    if (n == 1) return 0;
    while ((unsigned)p >= (unsigned)n) p = p < 0 ? -p - 1 + delta : 2 * n - 1 - p - delta;
    return p;
}

__device__ __forceinline__ int clamp16(int v) { return max(-32768, min(32767, v)); }

// 1/32-px source coordinates of output pixel (px, py) for layer g
__device__ __forceinline__ void mb_coords(const McsLayer& g, int px, int py, int& X, int& Y) {
    const int xl = px - g.ox, yl = py - g.oy;
    X = xl * 32;
    Y = yl * 32;
    if (g.kind != MCS_LAYER_COPY) layer_coords(g, xl, yl, X, Y);
}

// pyrUp taps of destination index d along an axis whose source has n values: the source is zero-inserted
// to 2n and convolved with [1 4 6 4 1] under BORDER_REFLECT_101, which keeps the parity of an index.
__device__ __forceinline__ void up_taps(int d, int n, int (&idx)[3], int (&wt)[3]) {
    const bool even = (d & 1) == 0;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        const int m = even ? 2 * t - 2 : 2 * t - 1;
        idx[t] = refl(d + m, 2 * n, 1) >> 1;
        wt[t] = even ? (t == 1 ? 6 : 1) : (t == 2 ? 0 : 4);
    }
}

// pyrUp of an int16 plane (sw x sh, C channels) at destination (x, y): (s + 32) >> 6, saturated
template <int C>
__device__ __forceinline__ void pyr_up_at(const int16_t* __restrict__ p, int sw, int sh, int x, int y, int (&out)[C]) {
    int ry[3], wy[3], rx[3], wx[3];
    up_taps(y, sh, ry, wy);
    up_taps(x, sw, rx, wx);
    int s[C];
#pragma unroll
    for (int c = 0; c < C; ++c) s[c] = 32;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        if (wy[a] == 0) continue;
        const int16_t* row = p + (long long)ry[a] * sw * C;
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            if (wx[b] == 0) continue;
            const int w = wy[a] * wx[b];
#pragma unroll
            for (int c = 0; c < C; ++c) s[c] += w * (int)__ldg(row + rx[b] * C + c);
        }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = clamp16(s[c] >> 6);
}

// Level 0 of every camera of the sub-batch: grid.z = camera + n_cams * frame.  GAIN: the rounded sample goes through
// the layer's exposure table.
template <int C, bool GAIN>
__global__ void __launch_bounds__(MB_BX * MB_BY) mb_level0_kernel(const __grid_constant__ MbArgs a) {
    const int j = blockIdx.z % a.n_cams, f = blockIdx.z / a.n_cams;
    const MbCam& c = a.cam[j];
    const int x = blockIdx.x * MB_BX + threadIdx.x, y = blockIdx.y * MB_BY + threadIdx.y;
    if (x >= c.bw || y >= c.bh) return;
    const int px = c.x0 + refl(c.tlx + x - c.x0, c.x1 - c.x0, 0);   // copyMakeBorder(BORDER_REFLECT)
    const int py = c.y0 + refl(c.tly + y - c.y0, c.y1 - c.y0, 0);
    const McsLayer& g = a.g[c.k];
    int X, Y;
    mb_coords(g, px, py, X, Y);
    const int sx = sat16(X >> 5), sy = sat16(Y >> 5), ax = X & 31, ay = Y & 31;
    const bool x0in = (unsigned)sx < (unsigned)g.src_w, x1in = (unsigned)(sx + 1) < (unsigned)g.src_w;
    const bool y0in = (unsigned)sy < (unsigned)g.src_h, y1in = (unsigned)(sy + 1) < (unsigned)g.src_h;
    const long long pitch = a.pitch[c.k];
    const uint8_t* r0 = a.src[c.k] + (long long)f * a.frame_stride[c.k] + (long long)sy * pitch + (long long)sx * C;
    const int w00 = (32 - ay) * (32 - ax) * 32, w01 = (32 - ay) * ax * 32, w10 = ay * (32 - ax) * 32, w11 = ay * ax * 32;
    int16_t* out = a.ws_cam + (long long)f * a.cam_elems + a.off[j][0] + ((long long)y * c.bw + x) * C;
#pragma unroll
    for (int ch = 0; ch < C; ++ch) {   // the overwrite sample: taps outside the source read 0
        int s = 16384;
        if (y0in && x0in) s += w00 * (int)__ldg(r0 + ch);
        if (y0in && x1in) s += w01 * (int)__ldg(r0 + C + ch);
        if (y1in && x0in) s += w10 * (int)__ldg(r0 + pitch + ch);
        if (y1in && x1in) s += w11 * (int)__ldg(r0 + pitch + C + ch);
        out[ch] = GAIN ? (int16_t)__ldg(a.lut + c.k * 256 + (s >> 15)) : (int16_t)(s >> 15);
    }
}

// Plan time: level 0 of every camera's weight pyramid, w + (w != 0) inside the rectangle, 0 in the border; w is the
// weight sample, or with Voronoi seams the seam-cut weight the plan holds.
__global__ void __launch_bounds__(MB_BX * MB_BY) mb_weight0_kernel(const __grid_constant__ MbArgs a) {
    const int j = blockIdx.z;
    const MbCam& c = a.cam[j];
    const int x = blockIdx.x * MB_BX + threadIdx.x, y = blockIdx.y * MB_BY + threadIdx.y;
    if (x >= c.bw || y >= c.bh) return;
    const int px = c.tlx + x, py = c.tly + y;
    int w = 0;
    if (px >= c.x0 && px < c.x1 && py >= c.y0 && py < c.y1) {
        if (a.seam[c.k]) {
            w = a.seam[c.k][(long long)(py - c.y0) * (c.x1 - c.x0) + px - c.x0];
        } else {
            const McsLayer& g = a.g[c.k];
            int X, Y;
            mb_coords(g, px, py, X, Y);
            w = weight_sample(a.wmap[c.k], g.src_w, g.src_h, X, Y);
        }
        w += w != 0 ? 1 : 0;
    }
    a.wpyr[a.woff[j][0] + (long long)y * c.bw + x] = (int16_t)w;
}

// pyrDown from level i to i + 1 of every camera: the frames' image pyramids (WEIGHTS = false, grid.z =
// camera + n_cams * frame) or the plan's weight pyramids (WEIGHTS = true, C = 1, grid.z = camera).
template <int C, bool WEIGHTS>
__global__ void __launch_bounds__(MB_BX * MB_BY) mb_pyrdown_kernel(const __grid_constant__ MbArgs a, int i) {
    const int j = blockIdx.z % a.n_cams, f = blockIdx.z / a.n_cams;
    const MbCam& c = a.cam[j];
    const int sw = c.bw >> i, sh = c.bh >> i, dw = sw >> 1, dh = sh >> 1;
    const int x = blockIdx.x * MB_BX + threadIdx.x, y = blockIdx.y * MB_BY + threadIdx.y;
    if (x >= dw || y >= dh) return;
    const int16_t* s = WEIGHTS ? a.wpyr + a.woff[j][i] : a.ws_cam + (long long)f * a.cam_elems + a.off[j][i];
    int16_t* d = WEIGHTS ? a.wpyr + a.woff[j][i + 1] : a.ws_cam + (long long)f * a.cam_elems + a.off[j][i + 1];
    const int k5[5] = {1, 4, 6, 4, 1};
    int cx[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) cx[q] = refl(2 * x + q - 2, sw, 1) * C;
    int acc[C];
#pragma unroll
    for (int ch = 0; ch < C; ++ch) acc[ch] = 128;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
        const int16_t* row = s + (long long)refl(2 * y + r - 2, sh, 1) * sw * C;
        int rs[C];
#pragma unroll
        for (int ch = 0; ch < C; ++ch) rs[ch] = 0;
#pragma unroll
        for (int q = 0; q < 5; ++q)
#pragma unroll
            for (int ch = 0; ch < C; ++ch) rs[ch] += k5[q] * (int)__ldg(row + cx[q] + ch);
#pragma unroll
        for (int ch = 0; ch < C; ++ch) acc[ch] += k5[r] * rs[ch];
    }
    int16_t* o = d + ((long long)y * dw + x) * C;
#pragma unroll
    for (int ch = 0; ch < C; ++ch) o[ch] = (int16_t)clamp16(acc[ch] >> 8);
}

// Plan time: the weight sums of level i (int16, wrapping like OpenCV's running sum).
__global__ void __launch_bounds__(MB_BX * MB_BY) mb_wsum_kernel(const __grid_constant__ MbArgs a, int i) {
    const int lw = a.roi_w >> i, lh = a.roi_h >> i;
    const int x = blockIdx.x * MB_BX + threadIdx.x, y = blockIdx.y * MB_BY + threadIdx.y;
    if (x >= lw || y >= lh) return;
    int s = 0;
    for (int j = 0; j < a.n_cams; ++j) {
        const MbCam& c = a.cam[j];
        const int lx = x - (c.tlx >> i), ly = y - (c.tly >> i), sw = c.bw >> i, sh = c.bh >> i;
        if ((unsigned)lx < (unsigned)sw && (unsigned)ly < (unsigned)sh) s += a.wpyr[a.woff[j][i] + (long long)ly * sw + lx];
    }
    a.wsum[a.soff[i] + (long long)y * lw + x] = (int16_t)s;
}

// Level i of the panorama for every frame of the sub-batch (grid.z = frame), levels n down to 0.
template <int C>
__global__ void __launch_bounds__(MB_BX * MB_BY) mb_blend_kernel(const __grid_constant__ MbArgs a, int i) {
    const int f = blockIdx.z;
    const int lw = a.roi_w >> i, lh = a.roi_h >> i;
    const int x = blockIdx.x * MB_BX + threadIdx.x, y = blockIdx.y * MB_BY + threadIdx.y;
    if (i == 0 ? (x >= a.out_w || y >= a.out_h) : (x >= lw || y >= lh)) return;
    const bool top = i == a.n_bands;
    const int16_t* cams = a.ws_cam + (long long)f * a.cam_elems;
    int acc[C];
#pragma unroll
    for (int ch = 0; ch < C; ++ch) acc[ch] = 0;
    for (int j = 0; j < a.n_cams; ++j) {
        const MbCam& c = a.cam[j];
        const int lx = x - (c.tlx >> i), ly = y - (c.tly >> i), sw = c.bw >> i, sh = c.bh >> i;
        if ((unsigned)lx >= (unsigned)sw || (unsigned)ly >= (unsigned)sh) continue;
        const int w = a.wpyr[a.woff[j][i] + (long long)ly * sw + lx];
        if (w == 0) continue;   // (L * 0) >> 8 adds nothing
        const int16_t* gp = cams + a.off[j][i] + ((long long)ly * sw + lx) * C;
        int lap[C];
#pragma unroll
        for (int ch = 0; ch < C; ++ch) lap[ch] = __ldg(gp + ch);
        if (!top) {
            int up[C];
            pyr_up_at<C>(cams + a.off[j][i + 1], sw >> 1, sh >> 1, lx, ly, up);
#pragma unroll
            for (int ch = 0; ch < C; ++ch) lap[ch] = clamp16(lap[ch] - up[ch]);
        }
#pragma unroll
        for (int ch = 0; ch < C; ++ch) acc[ch] += (lap[ch] * w) >> 8;
    }
    const int S = a.wsum[a.soff[i] + (long long)y * lw + x];
    int r[C];
#pragma unroll
    for (int ch = 0; ch < C; ++ch) r[ch] = (int16_t)((int)(int16_t)acc[ch] * 256 / (S + 1));
    if (!top) {
        int up[C];
        pyr_up_at<C>(a.ws_pan + (long long)f * a.pan_elems + a.poff[i + 1], lw >> 1, lh >> 1, x, y, up);
#pragma unroll
        for (int ch = 0; ch < C; ++ch) r[ch] = clamp16(r[ch] + up[ch]);
    }
    if (i > 0) {
        int16_t* o = a.ws_pan + (long long)f * a.pan_elems + a.poff[i] + ((long long)y * lw + x) * C;
#pragma unroll
        for (int ch = 0; ch < C; ++ch) o[ch] = (int16_t)r[ch];
        return;
    }
    uint8_t* o = a.dst + (long long)f * a.dst_frame_stride + (long long)y * a.dst_pitch + (long long)x * C;
#pragma unroll
    for (int ch = 0; ch < C; ++ch) o[ch] = S > 0 ? (uint8_t)max(0, min(255, r[ch])) : (uint8_t)0;
}

static dim3 mb_grid(int w, int h, int z) { return dim3((w + MB_BX - 1) / MB_BX, (h + MB_BY - 1) / MB_BY, z); }

void mcs_multiband_free(mcs_plan* plan) {
    McsMultiband* m = plan->mb;
    if (m) {
        cudaFree(m->a.wpyr);
        cudaFree(m->a.ws_cam);
        delete m;
    }
    plan->mb = nullptr;
    plan->mb_bands = 0;
}

int mcs_multiband_build(mcs_plan* plan, int bands) {
    mcs_multiband_free(plan);
    const int max_len = plan->out_w > plan->out_h ? plan->out_w : plan->out_h;
    // prepare(): the band count is clamped to ceil(log2 of the longer side), computed as OpenCV does
    int n = bands;
    if (max_len >= 1) {
        const int cap = (int)ceil(log((double)max_len) / log(2.0));
        n = n < cap ? n : cap;
    }
    const int s = 1 << n;
    McsMultiband* m = new McsMultiband;
    memset(m, 0, sizeof(*m));
    MbArgs& a = m->a;
    a.n_bands = n;
    a.out_w = plan->out_w;
    a.out_h = plan->out_h;
    a.roi_w = plan->out_w + (s - plan->out_w % s) % s;
    a.roi_h = plan->out_h + (s - plan->out_h % s) % s;
    a.channels = plan->channels;
    const int C = plan->channels;
    long long cam = 0, wts = 0;
    for (int k = 0; k < plan->n_layers; ++k) {
        const McsLayer& L = plan->layers[k];
        a.g[k] = L;
        a.wmap[k] = plan->d_cwmap[k];
        a.seam[k] = plan->seams_on ? plan->d_seam[k] : nullptr;
        MbCam c;
        c.k = k;
        c.x0 = L.rx0 > 0 ? L.rx0 : 0;
        c.y0 = L.ry0 > 0 ? L.ry0 : 0;
        c.x1 = L.rx1 < plan->out_w ? L.rx1 : plan->out_w;
        c.y1 = L.ry1 < plan->out_h ? L.ry1 : plan->out_h;
        if (c.x1 <= c.x0 || c.y1 <= c.y0) continue;   // an empty rectangle feeds nothing
        // feed(): the rectangle grown by 3 * 2^n, clipped to the ROI, aligned to 2^n, shifted back inside
        const int gap = 3 * s;
        int tlx = c.x0 - gap > 0 ? c.x0 - gap : 0, tly = c.y0 - gap > 0 ? c.y0 - gap : 0;
        int brx = c.x1 + gap < a.roi_w ? c.x1 + gap : a.roi_w, bry = c.y1 + gap < a.roi_h ? c.y1 + gap : a.roi_h;
        tlx = (tlx >> n) << n;
        tly = (tly >> n) << n;
        int wd = brx - tlx, ht = bry - tly;
        wd += (s - wd % s) % s;
        ht += (s - ht % s) % s;
        brx = tlx + wd;
        bry = tly + ht;
        const int dx = brx - a.roi_w > 0 ? brx - a.roi_w : 0, dy = bry - a.roi_h > 0 ? bry - a.roi_h : 0;
        c.tlx = tlx - dx;
        c.tly = tly - dy;
        c.bw = wd;
        c.bh = ht;
        const int j = a.n_cams++;
        a.cam[j] = c;
        for (int i = 0; i <= n; ++i) {
            const long long px = (long long)(wd >> i) * (ht >> i);
            a.off[j][i] = cam;
            a.woff[j][i] = wts;
            cam += px * C;
            wts += px;
        }
        m->max_bw = wd > m->max_bw ? wd : m->max_bw;
        m->max_bh = ht > m->max_bh ? ht : m->max_bh;
    }
    long long pan = 0, sums = 0;
    for (int i = 0; i <= n; ++i) {
        const long long px = (long long)(a.roi_w >> i) * (a.roi_h >> i);
        a.soff[i] = sums;
        sums += px;
        a.poff[i] = i == 0 ? 0 : pan;   // level 0 goes straight to the caller's output
        if (i > 0) pan += px * C;
    }
    a.cam_elems = cam;
    a.pan_elems = pan;
    m->ws_bytes = (size_t)MCS_MB_FRAMES * (size_t)(cam + pan) * sizeof(int16_t);
    plan->mb = m;
    plan->mb_bands = n;
    cudaError_t e = cudaMalloc(&a.wpyr, (size_t)(wts + sums + 1) * sizeof(int16_t));
    if (e == cudaSuccess) e = cudaMalloc(&a.ws_cam, m->ws_bytes + sizeof(int16_t));
    if (e == cudaSuccess) {
        a.wsum = a.wpyr + wts;
        a.ws_pan = a.ws_cam + (size_t)MCS_MB_FRAMES * cam;
        if (a.n_cams > 0) {
            mb_weight0_kernel<<<mb_grid(m->max_bw, m->max_bh, a.n_cams), dim3(MB_BX, MB_BY, 1)>>>(a);
            for (int i = 0; i < n; ++i)
                mb_pyrdown_kernel<1, true><<<mb_grid(m->max_bw >> (i + 1), m->max_bh >> (i + 1), a.n_cams),
                                             dim3(MB_BX, MB_BY, 1)>>>(a, i);
        }
        for (int i = 0; i <= n; ++i)
            mb_wsum_kernel<<<mb_grid(a.roi_w >> i, a.roi_h >> i, 1), dim3(MB_BX, MB_BY, 1)>>>(a, i);
        mcs_count_launch((a.n_cams > 0 ? n + 1 : 0) + n + 1);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    }
    if (e != cudaSuccess) {
        mcs_multiband_free(plan);
        mcs_set_error("mcs_plan_set_multiband: %s", cudaGetErrorString(e));
        return MCS_ERR_CUDA;
    }
    return MCS_OK;
}

template <int C>
static void mb_launch_batch(const McsMultiband* m, const MbArgs& a, int nf, cudaStream_t stream) {
    const dim3 block(MB_BX, MB_BY, 1);
    const int n = a.n_bands;
    if (a.n_cams > 0) {
        if (a.lut)
            mb_level0_kernel<C, true><<<mb_grid(m->max_bw, m->max_bh, a.n_cams * nf), block, 0, stream>>>(a);
        else
            mb_level0_kernel<C, false><<<mb_grid(m->max_bw, m->max_bh, a.n_cams * nf), block, 0, stream>>>(a);
        for (int i = 0; i < n; ++i)
            mb_pyrdown_kernel<C, false><<<mb_grid(m->max_bw >> (i + 1), m->max_bh >> (i + 1), a.n_cams * nf), block, 0,
                                          stream>>>(a, i);
    }
    for (int i = n; i >= 0; --i) {
        const int w = i == 0 ? a.out_w : a.roi_w >> i, h = i == 0 ? a.out_h : a.roi_h >> i;
        mb_blend_kernel<C><<<mb_grid(w, h, nf), block, 0, stream>>>(a, i);
    }
    mcs_count_launch((a.n_cams > 0 ? n + 1 : 0) + n + 1);
}

int mcs_launch_multiband(const mcs_plan* plan, const uint8_t* const* src, const int64_t* pitch, const int64_t* fstride,
                         int n_frames, uint8_t* dst, int64_t dst_pitch, int64_t dst_frame_stride, cudaStream_t stream) {
    const McsMultiband* m = plan->mb;
    MbArgs a = m->a;
    a.dst_pitch = dst_pitch;
    a.dst_frame_stride = dst_frame_stride;
    a.lut = plan->gains_on ? plan->d_gain_lut : nullptr;
    for (int f0 = 0; f0 < n_frames; f0 += MCS_MB_FRAMES) {
        const int nf = n_frames - f0 < MCS_MB_FRAMES ? n_frames - f0 : MCS_MB_FRAMES;
        for (int k = 0; k < plan->n_layers; ++k) {
            const long long fs = (fstride && n_frames > 1) ? fstride[k] : 0;
            a.src[k] = src[k] + (long long)f0 * fs;
            a.pitch[k] = pitch[k];
            a.frame_stride[k] = fs;
        }
        a.dst = dst + (long long)f0 * dst_frame_stride;
        switch (plan->channels) {
            case 1: mb_launch_batch<1>(m, a, nf, stream); break;
            case 3: mb_launch_batch<3>(m, a, nf, stream); break;
            default: mb_launch_batch<4>(m, a, nf, stream); break;
        }
        MCS_CHECK_CUDA(cudaGetLastError());
    }
    return MCS_OK;
}
