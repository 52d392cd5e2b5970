// Camera-weighted blend (mcs_plan_set_camera_weights, sm_100a).  Specification:
// oracle/camera_weight_model.py.  For output pixel p and layer k of the plan:
//   reach_k  p lies in the layer's visible rectangle
//   v_k      what the layer produces at p in overwrite mode (COPY: the source pixel; WARP / REMAP: the
//            fixed-point bilinear sample, BORDER_CONSTANT 0)
//   w_k      the same sample - same coordinates, taps and rounding - of the camera's uint8 weight map
//            (one byte per source pixel; no map = 255 everywhere)
//   contributors {k : reach_k and w_k > 0},  S = sum of their w_k
//   out = (sum w_k * v_k + S / 2) / S per channel (integer division), 0 where S == 0
// With one contributor that is v_k itself, so the single-contributor pixels skip the division.
//
// One thread per output pixel, the frames of the launch looped inside the thread (the mould of
// mcs_stitch_gather_frames_kernel, mcs_stitch.cu).  Everything that does not depend on the frame -
// rectangle tests, float64 coordinates, the weight sample, S and its reciprocal - runs once per
// pixel and launch; up to MCS_CW_MAX_CONTRIB contributors stay in registers.  Per frame only the
// taps, the integer samples, the weighted sum and one multiply-high remain.
#include "mcs_device.cuh"

#include <string.h>

struct CwArgs {
    McsLayer g[MCS_MAX_LAYERS];
    const uint8_t* src[MCS_MAX_LAYERS];
    long long pitch[MCS_MAX_LAYERS];
    long long frame_stride[MCS_MAX_LAYERS];
    const uint8_t* wmap[MCS_MAX_LAYERS];   // device, src_h x src_w bytes, or nullptr = 255 everywhere
    uint8_t* dst;
    long long dst_pitch;
    long long dst_frame_stride;
    int n_layers;
    int out_w, out_h;
    int n_frames;
};

#define CW_BX 64
#define CW_BY 4
#define CW_FRAMES 16   // frames per thread (grid.z covers the rest)

// One contributor: tap address of the launch's first frame, packed 16-bit tap weights for IDP.2A,
// and meta = tap-inside flags (bits 0..3: 00, 01, 10, 11) | word path (bit 4) | layer << 8 | w_k << 16.
struct Contrib {
    const uint8_t* r0;
    uint32_t wu, wl;
    uint32_t meta;
};

template <int C, bool WORDS>
__device__ __forceinline__ void contrib_sample(const CwArgs& a, const Contrib& q, int f, int (&v)[C]) {
    const int k = (q.meta >> 8) & 0xff;
    const long long pitch = a.pitch[k];
    const uint8_t* r0 = q.r0 + (long long)f * a.frame_stride[k];
    if (WORDS && (q.meta & 16u)) {
        const uint32_t phase = (uint32_t)(reinterpret_cast<uintptr_t>(r0) & 3u), sh = phase * 8u;
        const uint32_t* q0 = reinterpret_cast<const uint32_t*>(r0 - phase);
        const uint32_t* q1 = q0 + (pitch >> 2);
        const bool n1 = phase + 2 * C > 4, n2 = phase + 2 * C > 8;
        const uint32_t u0 = __ldg(q0), u1 = n1 ? __ldg(q0 + 1) : 0u, u2 = n2 ? __ldg(q0 + 2) : 0u;
        const uint32_t w0 = __ldg(q1), w1 = n1 ? __ldg(q1 + 1) : 0u, w2 = n2 ? __ldg(q1 + 2) : 0u;
        const uint32_t lo0 = __funnelshift_r(u0, u1, sh), hi0 = __funnelshift_r(u1, u2, sh);
        const uint32_t lo1 = __funnelshift_r(w0, w1, sh), hi1 = __funnelshift_r(w1, w2, sh);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const uint32_t sel = (uint32_t)c | ((uint32_t)(C + c) << 4);
            const uint32_t tu = __byte_perm(lo0, hi0, sel), tl = __byte_perm(lo1, hi1, sel);
            v[c] = (int)(__dp2a_lo(q.wl, tl, __dp2a_lo(q.wu, tu, 16384u)) >> 15);
        }
        return;
    }
    uint32_t p0[C], p1[C];   // tap pairs of the upper and lower row: byte 0 = left tap, byte 1 = right tap
#pragma unroll
    for (int c = 0; c < C; ++c) p0[c] = p1[c] = 0u;
    const uint32_t t = q.meta;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        if (t & 1u) p0[c] = __ldg(r0 + c);
        if (t & 2u) p0[c] |= (uint32_t)__ldg(r0 + C + c) << 8;
        if (t & 4u) p1[c] = __ldg(r0 + pitch + c);
        if (t & 8u) p1[c] |= (uint32_t)__ldg(r0 + pitch + C + c) << 8;
    }
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = (int)(__dp2a_lo(q.wl, p1[c], __dp2a_lo(q.wu, p0[c], 16384u)) >> 15);
}

template <int C, bool WORDS>
__global__ void __launch_bounds__(CW_BX * CW_BY)
mcs_stitch_weighted_kernel(const __grid_constant__ CwArgs a) {
    const int x = blockIdx.x * CW_BX + threadIdx.x;
    const int y = blockIdx.y * CW_BY + threadIdx.y;
    if (x >= a.out_w || y >= a.out_h) return;
    const int f0 = blockIdx.z * CW_FRAMES;
    const int n_fr = min(CW_FRAMES, a.n_frames - f0);
    uint8_t* out = a.dst + (long long)f0 * a.dst_frame_stride + (long long)y * a.dst_pitch + (long long)x * C;

    Contrib q[MCS_CW_MAX_CONTRIB];
    int n = 0;
    uint32_t S = 0;
    for (int k = 0; k < a.n_layers && n < MCS_CW_MAX_CONTRIB; ++k) {
        const McsLayer& g = a.g[k];
        if (x < g.rx0 || x >= g.rx1 || y < g.ry0 || y >= g.ry1) continue;
        const int xl = x - g.ox, yl = y - g.oy;
        int X, Y;
        if (g.kind == MCS_LAYER_COPY) {
            X = xl * 32;
            Y = yl * 32;
        } else {
            layer_coords(g, xl, yl, X, Y);
        }
        const int wk = weight_sample(a.wmap[k], g.src_w, g.src_h, X, Y);
        if (wk == 0) continue;
        const int sx = sat16(X >> 5), sy = sat16(Y >> 5), ax = X & 31, ay = Y & 31;
        const bool x0in = (unsigned)sx < (unsigned)g.src_w, x1in = (unsigned)(sx + 1) < (unsigned)g.src_w;
        const bool y0in = (unsigned)sy < (unsigned)g.src_h, y1in = (unsigned)(sy + 1) < (unsigned)g.src_h;
        const uint32_t taps = (y0in && x0in ? 1u : 0u) | (y0in && x1in ? 2u : 0u) | (y1in && x0in ? 4u : 0u) |
                              (y1in && x1in ? 8u : 0u);
        const bool words = WORDS && taps == 15u && sy + 2 < g.src_h;
        Contrib c;
        // taps outside the source are never dereferenced, so the address may point anywhere
        c.r0 = a.src[k] + (long long)f0 * a.frame_stride[k] + (long long)sy * a.pitch[k] + (long long)sx * C;
        c.wu = (uint32_t)((32 - ay) * (32 - ax) * 32) | ((uint32_t)((32 - ay) * ax * 32) << 16);
        c.wl = (uint32_t)(ay * (32 - ax) * 32) | ((uint32_t)(ay * ax * 32) << 16);
        c.meta = taps | (words ? 16u : 0u) | ((uint32_t)k << 8) | ((uint32_t)wk << 16);
#pragma unroll
        for (int j = 0; j < MCS_CW_MAX_CONTRIB; ++j)   // constant indices: the slots stay in registers
            if (j == n) q[j] = c;
        S += (uint32_t)wk;
        ++n;
    }
    // ceil(2^32 / S): __umulhi(num, m) == num / S for 2 <= S <= 1020 and num <= 255 * S + S / 2
    const uint32_t m = S > 1 ? 0xffffffffu / S + 1u : 0u;
    const uint32_t half = S >> 1;

    for (int f = 0; f < n_fr; ++f, out += a.dst_frame_stride) {
        int r[C];
        if (n == 0) {
#pragma unroll
            for (int c = 0; c < C; ++c) r[c] = 0;
        } else if (n == 1) {
            contrib_sample<C, WORDS>(a, q[0], f, r);
        } else {
            uint32_t acc[C];
#pragma unroll
            for (int c = 0; c < C; ++c) acc[c] = half;
#pragma unroll
            for (int j = 0; j < MCS_CW_MAX_CONTRIB; ++j) {
                if (j < n) {
                    int v[C];
                    contrib_sample<C, WORDS>(a, q[j], f, v);
                    const uint32_t wk = q[j].meta >> 16;
#pragma unroll
                    for (int c = 0; c < C; ++c) acc[c] += wk * (uint32_t)v[c];
                }
            }
#pragma unroll
            for (int c = 0; c < C; ++c) r[c] = (int)__umulhi(acc[c], m);
        }
#pragma unroll
        for (int c = 0; c < C; ++c) out[c] = (uint8_t)r[c];
    }
}

// Plan-time counter: per layer, the output pixels it contributes to, and the most contributors any
// pixel has (all of them, also past MCS_CW_MAX_CONTRIB: the setter refuses such rigs).  Blocks of
// 32 x 16 pixels; whole warps stay alive for the warp-level merge.
__global__ void __launch_bounds__(512)
mcs_camera_weights_count_kernel(const __grid_constant__ CwArgs a, unsigned long long* __restrict__ contrib,
                                unsigned* __restrict__ max_count) {
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 16 + threadIdx.y;
    const bool live = x < a.out_w && y < a.out_h;
    int n = 0;
    for (int k = 0; k < a.n_layers; ++k) {
        const McsLayer& g = a.g[k];
        bool in = live && x >= g.rx0 && x < g.rx1 && y >= g.ry0 && y < g.ry1;
        if (in) {
            const int xl = x - g.ox, yl = y - g.oy;
            int X = xl * 32, Y = yl * 32;
            if (g.kind != MCS_LAYER_COPY) layer_coords(g, xl, yl, X, Y);
            in = weight_sample(a.wmap[k], g.src_w, g.src_h, X, Y) > 0;
        }
        n += in ? 1 : 0;
        const unsigned ballot = __ballot_sync(0xffffffffu, in);
        if (threadIdx.x == 0 && ballot) atomicAdd(contrib + k, (unsigned long long)__popc(ballot));
    }
    const unsigned most = __reduce_max_sync(0xffffffffu, (unsigned)n);
    if (threadIdx.x == 0 && most) atomicMax(max_count, most);
}

static void fill_cw_args(const mcs_plan* plan, CwArgs& a) {
    memset(&a, 0, sizeof(a));
    a.n_layers = plan->n_layers;
    a.out_w = plan->out_w;
    a.out_h = plan->out_h;
    for (int k = 0; k < plan->n_layers; ++k) {
        a.g[k] = plan->layers[k];
        a.wmap[k] = plan->d_cwmap[k];
    }
}

int mcs_camera_weights_count(const mcs_plan* plan, long long* contrib, int* max_count) {
    unsigned long long* d = nullptr;
    MCS_CHECK_CUDA(cudaMalloc(&d, sizeof(unsigned long long) * MCS_MAX_LAYERS + sizeof(unsigned)));
    unsigned* d_max = reinterpret_cast<unsigned*>(d + MCS_MAX_LAYERS);
    cudaError_t e = cudaMemset(d, 0, sizeof(unsigned long long) * MCS_MAX_LAYERS + sizeof(unsigned));
    if (e == cudaSuccess && plan->out_w > 0 && plan->out_h > 0) {
        CwArgs a;
        fill_cw_args(plan, a);
        const dim3 grid((plan->out_w + 31) / 32, (plan->out_h + 15) / 16, 1);
        mcs_camera_weights_count_kernel<<<grid, dim3(32, 16, 1)>>>(a, d, d_max);
        mcs_count_launch(1);
        e = cudaGetLastError();
    }
    unsigned long long h[MCS_MAX_LAYERS];
    unsigned hm = 0;
    if (e == cudaSuccess) e = cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(&hm, d_max, sizeof(hm), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) {
        mcs_set_error("mcs_plan_set_camera_weights: %s", cudaGetErrorString(e));
        return MCS_ERR_CUDA;
    }
    for (int k = 0; k < plan->n_layers; ++k) contrib[k] = (long long)h[k];
    *max_count = (int)hm;
    return MCS_OK;
}

int mcs_launch_weighted(const mcs_plan* plan, const uint8_t* const* src, const int64_t* pitch,
                        const int64_t* fstride, int n_frames, uint8_t* dst, int64_t dst_pitch,
                        int64_t dst_frame_stride, cudaStream_t stream) {
    CwArgs a;
    fill_cw_args(plan, a);
    a.n_frames = n_frames;
    a.dst = dst;
    a.dst_pitch = dst_pitch;
    a.dst_frame_stride = dst_frame_stride;
    bool words = true;   // every base, pitch and frame stride a multiple of 4 bytes: taps as aligned words
    for (int k = 0; k < plan->n_layers; ++k) {
        a.src[k] = src[k];
        a.pitch[k] = pitch[k];
        a.frame_stride[k] = (fstride && n_frames > 1) ? fstride[k] : 0;
        words = words && ((reinterpret_cast<uintptr_t>(a.src[k]) | (uintptr_t)a.pitch[k] | (uintptr_t)a.frame_stride[k]) & 3u) == 0;
    }
    dim3 block(CW_BX, CW_BY, 1);
    dim3 grid((plan->out_w + CW_BX - 1) / CW_BX, (plan->out_h + CW_BY - 1) / CW_BY, (n_frames + CW_FRAMES - 1) / CW_FRAMES);
    switch (plan->channels * 2 + (words ? 1 : 0)) {
        case 2: mcs_stitch_weighted_kernel<1, false><<<grid, block, 0, stream>>>(a); break;
        case 3: mcs_stitch_weighted_kernel<1, true><<<grid, block, 0, stream>>>(a); break;
        case 6: mcs_stitch_weighted_kernel<3, false><<<grid, block, 0, stream>>>(a); break;
        case 7: mcs_stitch_weighted_kernel<3, true><<<grid, block, 0, stream>>>(a); break;
        case 8: mcs_stitch_weighted_kernel<4, false><<<grid, block, 0, stream>>>(a); break;
        default: mcs_stitch_weighted_kernel<4, true><<<grid, block, 0, stream>>>(a); break;
    }
    mcs_count_launch(1);
    MCS_CHECK_CUDA(cudaGetLastError());
    return MCS_OK;
}
