// Voronoi seam masks for the multi-band blend (mcs_plan_set_voronoi_seams, sm_100a): OpenCV's
// cv::detail::VoronoiSeamFinder run on the cameras' weight samples w_k.  Specification:
// oracle/seam_model.py.  Plan time only; integer only.
//
// The plan keeps one u8 plane per fed layer (a layer with a non-empty clipped rectangle), the size of that
// rectangle: the seam-cut weights, which mb_weight0_kernel then reads instead of sampling the map.
//
//   1. seam_fill_kernel   one launch: every plane = the weight sample w_k (the sample mb_weight0_kernel takes)
//   2. per overlapping pair (i, j), i < j in feed order, two launches on the submask (the overlap ROI grown by
//      MCS_SEAM_GAP, reading 0 outside each plane), each pair cutting the planes the earlier pairs left:
//      seam_rows_kernel  one block per submask row: u1 = (s1 != 0) & (s2 == 0), u2 likewise, and the 1-D
//                        distance along the row to the nearest pixel of each (a chunk per thread, the carries
//                        across chunks by a block scan); records whether u1 / u2 has any pixel
//      seam_cols_kernel  one thread per submask column: min(h, prev + 1) down and up gives the exact L1
//                        distance (what distanceTransform(DIST_L1, 3) computes), the empty-plane rule
//                        MCS_SEAM_EMPTY + min(y + 1, x + 1, H - y, W - x) where u has no pixel; inside the ROI
//                        the pixel is zeroed in plane j where d1 < d2, otherwise in plane i
// A submask of W + H < MCS_SEAM_EMPTY keeps every real distance below MCS_SEAM_EMPTY, so the distances travel
// as uint16 (65535 = no pixel of u in the row / column so far); larger plans are refused.
#include "mcs_device.cuh"

#include <string.h>

#define MCS_SEAM_GAP 10        // the overlap ROI grows by this much on every side into the submask
#define MCS_SEAM_EMPTY 32768   // OpenCV's INT_MAX border after the float conversion; W + H must stay below it
#define SEAM_ROW_THREADS 128
#define SEAM_COL_THREADS 128
#define SEAM_NONE 65535
#define SEAM_BX 32
#define SEAM_BY 8

struct SeamFill {
    McsLayer g[MCS_MAX_LAYERS];
    const uint8_t* wmap[MCS_MAX_LAYERS];
    uint8_t* plane[MCS_MAX_LAYERS];
    int4 rect[MCS_MAX_LAYERS];   // clipped rectangle {x0, y0, x1, y1}
    int layer[MCS_MAX_LAYERS];   // fed layers in feed order
};

struct SeamPair {
    uint8_t* m[2];          // planes of cameras i and j
    int pw[2], ph[2];       // their sizes
    int ox[2], oy[2];       // submask origin in each plane's coordinates
    int W, H;               // submask size
    uint16_t* d[2];         // W x H distances of u1 / u2 (row pass, then the column pass in place)
    int* any;               // [2]: u1 / u2 has a pixel
};

// Plan time: every plane = the weight sample of its layer (grid.z = fed layer).
__global__ void __launch_bounds__(SEAM_BX * SEAM_BY) seam_fill_kernel(const __grid_constant__ SeamFill a) {
    const int k = a.layer[blockIdx.z];
    const int4 r = a.rect[k];
    const int x = blockIdx.x * SEAM_BX + threadIdx.x, y = blockIdx.y * SEAM_BY + threadIdx.y;
    if (x >= r.z - r.x || y >= r.w - r.y) return;
    const McsLayer& g = a.g[k];
    const int xl = r.x + x - g.ox, yl = r.y + y - g.oy;
    int X = xl * 32, Y = yl * 32;
    if (g.kind != MCS_LAYER_COPY) layer_coords(g, xl, yl, X, Y);
    a.plane[k][(long long)y * (r.z - r.x) + x] = (uint8_t)weight_sample(a.wmap[k], g.src_w, g.src_h, X, Y);
}

__device__ __forceinline__ bool seam_set(const SeamPair& p, int c, int x, int y) {
    const int px = p.ox[c] + x, py = p.oy[c] + y;
    return (unsigned)px < (unsigned)p.pw[c] && (unsigned)py < (unsigned)p.ph[c] &&
           p.m[c][(long long)py * p.pw[c] + px] != 0;
}

// u1 / u2 at (x, y): a camera's non-zero pixel where the other camera is zero
__device__ __forceinline__ void seam_unique(const SeamPair& p, int x, int y, bool& u1, bool& u2) {
    const bool s1 = seam_set(p, 0, x, y), s2 = seam_set(p, 1, x, y);
    u1 = s1 && !s2;
    u2 = s2 && !s1;
}

// One block per submask row: the 1-D distance along the row to the nearest pixel of u1 and of u2.
__global__ void __launch_bounds__(SEAM_ROW_THREADS) seam_rows_kernel(const __grid_constant__ SeamPair p) {
    __shared__ int lastx[2][SEAM_ROW_THREADS], firstx[2][SEAM_ROW_THREADS];
    const int y = blockIdx.x, t = threadIdx.x;
    const int chunk = (p.W + SEAM_ROW_THREADS - 1) / SEAM_ROW_THREADS;
    const int xa = min(p.W, t * chunk), xb = min(p.W, xa + chunk);
    int last[2] = {-1, -1}, first[2] = {p.W + SEAM_NONE, p.W + SEAM_NONE};
    for (int x = xa; x < xb; ++x) {
        bool u[2];
        seam_unique(p, x, y, u[0], u[1]);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            if (u[c]) last[c] = x;
            if (u[c] && first[c] > x) first[c] = x;
        }
    }
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        lastx[c][t] = last[c];
        firstx[c][t] = first[c];
    }
    __syncthreads();
    // inclusive scans: the last pixel at or before each chunk's end, the first at or after each chunk's start
    for (int off = 1; off < SEAM_ROW_THREADS; off <<= 1) {
        int l[2], f[2];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            l[c] = t >= off ? lastx[c][t - off] : -1;
            f[c] = t + off < SEAM_ROW_THREADS ? firstx[c][t + off] : p.W + SEAM_NONE;
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            lastx[c][t] = max(lastx[c][t], l[c]);
            firstx[c][t] = min(firstx[c][t], f[c]);
        }
        __syncthreads();
    }
    if (t == 0) {
#pragma unroll
        for (int c = 0; c < 2; ++c)
            if (lastx[c][SEAM_ROW_THREADS - 1] >= 0) atomicOr(p.any + c, 1);
    }
    int left[2], right[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        left[c] = t > 0 ? lastx[c][t - 1] : -1;
        right[c] = t + 1 < SEAM_ROW_THREADS ? firstx[c][t + 1] : p.W + SEAM_NONE;
    }
    uint16_t* row[2] = {p.d[0] + (long long)y * p.W, p.d[1] + (long long)y * p.W};
    for (int x = xa; x < xb; ++x) {   // distance to the left
        bool u[2];
        seam_unique(p, x, y, u[0], u[1]);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            if (u[c]) left[c] = x;
            row[c][x] = left[c] >= 0 ? (uint16_t)(x - left[c]) : (uint16_t)SEAM_NONE;
        }
    }
    for (int x = xb - 1; x >= xa; --x) {   // and to the right
        bool u[2];
        seam_unique(p, x, y, u[0], u[1]);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            if (u[c]) right[c] = x;
            row[c][x] = (uint16_t)min((int)row[c][x], min(right[c] - x, SEAM_NONE));
        }
    }
}

// One thread per submask column: exact L1 distances down and up the column, then the cut inside the ROI.
__global__ void __launch_bounds__(SEAM_COL_THREADS) seam_cols_kernel(const __grid_constant__ SeamPair p) {
    const int x = blockIdx.x * SEAM_COL_THREADS + threadIdx.x;
    if (x >= p.W) return;
    const int W = p.W, H = p.H;
    int f[2] = {SEAM_NONE, SEAM_NONE};
    for (int y = 0; y < H; ++y) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            uint16_t* d = p.d[c] + (long long)y * W + x;
            f[c] = min((int)*d, f[c] + 1);
            *d = (uint16_t)f[c];
        }
    }
    const bool any1 = p.any[0] != 0, any2 = p.any[1] != 0;
    const bool in_x = x >= MCS_SEAM_GAP && x < W - MCS_SEAM_GAP;
    int b[2] = {SEAM_NONE, SEAM_NONE};
    for (int y = H - 1; y >= 0; --y) {
#pragma unroll
        for (int c = 0; c < 2; ++c) b[c] = min((int)p.d[c][(long long)y * W + x], b[c] + 1);
        if (!in_x || y < MCS_SEAM_GAP || y >= H - MCS_SEAM_GAP) continue;
        const int border = MCS_SEAM_EMPTY + min(min(y + 1, x + 1), min(H - y, W - x));
        const int d1 = any1 ? b[0] : border, d2 = any2 ? b[1] : border;
        const int c = d1 < d2 ? 1 : 0;   // ties cut camera i
        p.m[c][(long long)(p.oy[c] + y) * p.pw[c] + p.ox[c] + x] = 0;
    }
}

void mcs_seams_fill(const mcs_plan* plan, uint8_t* const* planes) {
    SeamFill a;
    memset(&a, 0, sizeof(a));
    int n = 0, bw = 0, bh = 0;
    for (int k = 0; k < plan->n_layers; ++k) {
        const McsLayer& L = plan->layers[k];
        a.g[k] = L;
        a.wmap[k] = plan->d_cwmap[k];
        a.plane[k] = planes[k];
        const int x0 = L.rx0 > 0 ? L.rx0 : 0, y0 = L.ry0 > 0 ? L.ry0 : 0;
        const int x1 = L.rx1 < plan->out_w ? L.rx1 : plan->out_w, y1 = L.ry1 < plan->out_h ? L.ry1 : plan->out_h;
        a.rect[k] = make_int4(x0, y0, x1, y1);
        if (x1 > x0 && y1 > y0) {
            a.layer[n++] = k;
            bw = x1 - x0 > bw ? x1 - x0 : bw;
            bh = y1 - y0 > bh ? y1 - y0 : bh;
        }
    }
    if (n == 0) return;
    seam_fill_kernel<<<dim3((bw + SEAM_BX - 1) / SEAM_BX, (bh + SEAM_BY - 1) / SEAM_BY, n), dim3(SEAM_BX, SEAM_BY, 1)>>>(a);
    mcs_count_launch(1);
}

void mcs_seams_free(mcs_plan* plan) {
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) {
        if (plan->d_seam[k]) cudaFree(plan->d_seam[k]);
        plan->d_seam[k] = nullptr;
    }
    plan->seams_on = 0;
}

int mcs_seams_build(mcs_plan* plan) {
    SeamFill a;
    memset(&a, 0, sizeof(a));
    int n = 0;
    for (int k = 0; k < plan->n_layers; ++k) {
        const McsLayer& L = plan->layers[k];
        a.g[k] = L;
        a.wmap[k] = plan->d_cwmap[k];
        const int x0 = L.rx0 > 0 ? L.rx0 : 0, y0 = L.ry0 > 0 ? L.ry0 : 0;
        const int x1 = L.rx1 < plan->out_w ? L.rx1 : plan->out_w, y1 = L.ry1 < plan->out_h ? L.ry1 : plan->out_h;
        a.rect[k] = make_int4(x0, y0, x1, y1);
        if (x1 > x0 && y1 > y0) a.layer[n++] = k;   // an empty rectangle feeds nothing
    }
    // the pairs (overlapRoi) and the bound, before anything in the plan changes
    int pi[MCS_MAX_LAYERS * MCS_MAX_LAYERS / 2], pj[MCS_MAX_LAYERS * MCS_MAX_LAYERS / 2];
    int np = 0, max_w = 0, max_h = 0;
    long long max_px = 0;
    for (int u = 0; u < n; ++u)
        for (int v = u + 1; v < n; ++v) {
            const int4 r1 = a.rect[a.layer[u]], r2 = a.rect[a.layer[v]];
            const int rx0 = max(r1.x, r2.x), ry0 = max(r1.y, r2.y), rx1 = min(r1.z, r2.z), ry1 = min(r1.w, r2.w);
            if (rx0 >= rx1 || ry0 >= ry1) continue;
            const int W = rx1 - rx0 + 2 * MCS_SEAM_GAP, H = ry1 - ry0 + 2 * MCS_SEAM_GAP;
            if (W + H >= MCS_SEAM_EMPTY) {
                mcs_set_error("mcs_plan_set_voronoi_seams: layers %d and %d overlap in a %d x %d submask; W + H must stay "
                              "below %d", a.layer[u], a.layer[v], W, H, MCS_SEAM_EMPTY);
                return MCS_ERR_UNSUPPORTED;
            }
            pi[np] = a.layer[u];
            pj[np] = a.layer[v];
            ++np;
            max_w = W > max_w ? W : max_w;
            max_h = H > max_h ? H : max_h;
            max_px = (long long)W * H > max_px ? (long long)W * H : max_px;
        }
    mcs_seams_free(plan);
    uint16_t* scratch = nullptr;
    int* any = nullptr;
    cudaError_t e = cudaSuccess;
    int launches = 0;
    for (int u = 0; u < n && e == cudaSuccess; ++u) {
        const int4 r = a.rect[a.layer[u]];
        e = cudaMalloc(&plan->d_seam[a.layer[u]], (size_t)(r.z - r.x) * (r.w - r.y));
        a.plane[a.layer[u]] = plan->d_seam[a.layer[u]];
    }
    if (e == cudaSuccess && np > 0) e = cudaMalloc(&scratch, (size_t)2 * max_px * sizeof(uint16_t));
    if (e == cudaSuccess && np > 0) e = cudaMalloc(&any, (size_t)2 * np * sizeof(int));
    if (e == cudaSuccess && np > 0) e = cudaMemsetAsync(any, 0, (size_t)2 * np * sizeof(int), 0);
    if (e == cudaSuccess && n > 0) {
        int bw = 0, bh = 0;
        for (int u = 0; u < n; ++u) {
            const int4 r = a.rect[a.layer[u]];
            bw = r.z - r.x > bw ? r.z - r.x : bw;
            bh = r.w - r.y > bh ? r.w - r.y : bh;
        }
        seam_fill_kernel<<<dim3((bw + SEAM_BX - 1) / SEAM_BX, (bh + SEAM_BY - 1) / SEAM_BY, n), dim3(SEAM_BX, SEAM_BY, 1)>>>(a);
        ++launches;
        for (int q = 0; q < np; ++q) {
            SeamPair p;
            const int i = pi[q], j = pj[q];
            const int4 r1 = a.rect[i], r2 = a.rect[j];
            const int rx0 = max(r1.x, r2.x), ry0 = max(r1.y, r2.y), rx1 = min(r1.z, r2.z), ry1 = min(r1.w, r2.w);
            p.W = rx1 - rx0 + 2 * MCS_SEAM_GAP;
            p.H = ry1 - ry0 + 2 * MCS_SEAM_GAP;
            const int4 rr[2] = {r1, r2};
            const int kk[2] = {i, j};
            for (int c = 0; c < 2; ++c) {
                p.m[c] = plan->d_seam[kk[c]];
                p.pw[c] = rr[c].z - rr[c].x;
                p.ph[c] = rr[c].w - rr[c].y;
                p.ox[c] = rx0 - MCS_SEAM_GAP - rr[c].x;
                p.oy[c] = ry0 - MCS_SEAM_GAP - rr[c].y;
                p.d[c] = scratch + (size_t)c * max_px;
            }
            p.any = any + 2 * q;
            seam_rows_kernel<<<p.H, SEAM_ROW_THREADS>>>(p);
            seam_cols_kernel<<<(p.W + SEAM_COL_THREADS - 1) / SEAM_COL_THREADS, SEAM_COL_THREADS>>>(p);
            launches += 2;
        }
        mcs_count_launch(launches);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    }
    if (scratch) cudaFree(scratch);
    if (any) cudaFree(any);
    if (e != cudaSuccess) {
        mcs_seams_free(plan);
        mcs_set_error("mcs_plan_set_voronoi_seams: %s", cudaGetErrorString(e));
        return MCS_ERR_CUDA;
    }
    plan->seams_on = 1;
    return MCS_OK;
}
