// Graph-cut seam masks for the multi-band blend (mcs_plan_set_graphcut_seams, sm_100a): OpenCV's
// cv::detail::GraphCutSeamFinder("COST_COLOR") run on the cameras' weight samples w_k and the overwrite samples v_k
// of one frame-set.  Specification: oracle/graphcut_seam_model.py (find_graphcut).  Plan time only; integer only.
//
//   1. seam_fill_kernel (mcs_seams.cu)  every new plane = the weight sample w_k
//      gc_sample_kernel                 every fed layer's v_k over its clipped rectangle, 3 bytes a pixel (the sample
//                                       mb_level0_kernel takes, through the exposure tables when the plan has gains)
//   2. per overlapping pair (i, j), i < j in feed order, on the submask (the overlap ROI grown by MCS_GC_GAP, reading
//      0 outside each plane), each pair cutting the planes the earlier pairs left:
//      gc_caps_kernel    D(p) = sum_c (I1_c - I2_c)^2, the grid capacities D(p) + D(q) + 1 (+ MCS_GC_PENALTY where a
//                        mask of p or q is 0) and the terminal capacities MCS_GC_TERMINAL
//      an exact maximum flow by push-relabel, host-driven rounds of launches:
//        gc_label_init_kernel + gc_relax_kernel (repeated)  global relabel: exact residual distances to the terminal
//                        (breadth-first, as a relaxation of 32 x 32 tiles in shared memory until nothing changes)
//        gc_count_kernel  the active nodes (excess, finite label); none left ends the flow
//        gc_push_kernel + gc_pull_kernel, MCS_GC_ROUNDS times between global relabels: every active node pushes
//                        down admissible edges (its own residuals and excess only), then every node takes in what
//                        its neighbours pushed and relabels from the labels of the round (double-buffered)
//      gc_cut_kernel     inside the ROI: p in S with s1 != 0 is zeroed in plane j, p not in S with s2 != 0 in plane i
//
// The flow runs on the reversed network: it pushes from the sink terminals (s2 != 0) toward the source terminals
// (s1 != 0); the grid capacities are symmetric, so only the terminals swap.  The final global relabel then labels
// exactly the pixels that can reach the source terminals in the residual graph of the reversed flow, i.e. the pixels
// reachable from the source in the residual graph of the original one: S, the minimal source side of a minimum cut.
// Every maximum flow gives the same S, so the order of the pushes does not matter.  The largest edge is 391 151 and
// at most 1 574 604 can enter a node, so residuals and excesses are int32.
#include "mcs_device.cuh"

#include <string.h>

#define MCS_GC_GAP 10           // the overlap ROI grows by this much on every side into the submask
#define MCS_GC_TERMINAL 10000   // GraphCutSeamFinder's terminal_cost
#define MCS_GC_PENALTY 1000     // its bad_region_penalty: an edge touching a zero mask pixel
#define MCS_GC_ROUNDS 64        // push / pull rounds between global relabels
#define MCS_GC_RELAX 4          // relaxation launches per read-back of a global relabel
#define MCS_GC_MAX_ROUNDS (1 << 22)   // guard against a bug: far above anything a real submask takes
#define GC_BX 32
#define GC_BY 8
#define GC_TILE 32              // gc_relax_kernel: a 32 x 32 tile per block, 4 rows per thread

struct GcSample {
    McsLayer g[MCS_MAX_LAYERS];
    const uint8_t* src[MCS_MAX_LAYERS];
    long long pitch[MCS_MAX_LAYERS];
    uint8_t* img[MCS_MAX_LAYERS];   // 3 bytes a pixel over the clipped rectangle
    int4 rect[MCS_MAX_LAYERS];      // clipped rectangle {x0, y0, x1, y1}
    int layer[MCS_MAX_LAYERS];      // fed layers in feed order
    const uint8_t* lut;             // GAIN: per layer the 256-entry exposure table (mcs_exposure.cu)
};

struct GcPair {
    uint8_t* m[2];          // planes of cameras i and j
    const uint8_t* img[2];  // their samples, 3 bytes a pixel
    int pw[2], ph[2];       // their sizes
    int ox[2], oy[2];       // submask origin in each plane's coordinates
    int W, H, N;            // submask size; N = W * H is also the label of "cannot reach the terminal"
    int* e;                 // N excess
    int* h;                 // N labels
    int* h2;                // N labels of the next round
    int* rt;                // N residual to the terminal (the original source, s1 != 0)
    int* r;                 // 4 N residuals to the right, left, down and up neighbours
    int* out;               // 4 N what a round pushed that way
    int* flags;             // MCS_GC_RELAX change flags of a relaxation batch, then the active count
};

// Plan time: v_k of every fed layer (grid.z = fed layer): the overwrite sample, taps outside the source read 0;
// with GAIN its value in the layer's exposure table, the sample the blends then take.
template <bool GAIN>
__global__ void __launch_bounds__(GC_BX * GC_BY) gc_sample_kernel(const __grid_constant__ GcSample a) {
    const int k = a.layer[blockIdx.z];
    const int4 r = a.rect[k];
    const int x = blockIdx.x * GC_BX + threadIdx.x, y = blockIdx.y * GC_BY + threadIdx.y;
    if (x >= r.z - r.x || y >= r.w - r.y) return;
    const McsLayer& g = a.g[k];
    const int xl = r.x + x - g.ox, yl = r.y + y - g.oy;
    int X = xl * 32, Y = yl * 32;
    if (g.kind != MCS_LAYER_COPY) layer_coords(g, xl, yl, X, Y);
    const int sx = sat16(X >> 5), sy = sat16(Y >> 5), ax = X & 31, ay = Y & 31;
    const bool x0in = (unsigned)sx < (unsigned)g.src_w, x1in = (unsigned)(sx + 1) < (unsigned)g.src_w;
    const bool y0in = (unsigned)sy < (unsigned)g.src_h, y1in = (unsigned)(sy + 1) < (unsigned)g.src_h;
    const long long pitch = a.pitch[k];
    const uint8_t* r0 = a.src[k] + (long long)sy * pitch + (long long)sx * 3;
    const int w00 = (32 - ay) * (32 - ax) * 32, w01 = (32 - ay) * ax * 32, w10 = ay * (32 - ax) * 32, w11 = ay * ax * 32;
    uint8_t* out = a.img[k] + ((long long)y * (r.z - r.x) + x) * 3;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        int s = 16384;
        if (y0in && x0in) s += w00 * (int)__ldg(r0 + ch);
        if (y0in && x1in) s += w01 * (int)__ldg(r0 + 3 + ch);
        if (y1in && x0in) s += w10 * (int)__ldg(r0 + pitch + ch);
        if (y1in && x1in) s += w11 * (int)__ldg(r0 + pitch + 3 + ch);
        out[ch] = GAIN ? __ldg(a.lut + k * 256 + (s >> 15)) : (uint8_t)(s >> 15);
    }
}

__device__ __forceinline__ bool gc_inside(const GcPair& p, int c, int x, int y, long long& at) {
    const int px = p.ox[c] + x, py = p.oy[c] + y;
    at = (long long)py * p.pw[c] + px;
    return (unsigned)px < (unsigned)p.pw[c] && (unsigned)py < (unsigned)p.ph[c];
}

// submask pixel (x, y): s1 != 0, s2 != 0 and D
__device__ __forceinline__ void gc_pixel(const GcPair& p, int x, int y, bool& s1, bool& s2, int& d) {
    int v[2][3];
    bool s[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        long long at;
        const bool in = gc_inside(p, c, x, y, at);
        s[c] = in && p.m[c][at] != 0;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) v[c][ch] = in ? (int)p.img[c][at * 3 + ch] : 0;
    }
    s1 = s[0];
    s2 = s[1];
    d = 0;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) d += (v[0][ch] - v[1][ch]) * (v[0][ch] - v[1][ch]);
}

__device__ __forceinline__ bool gc_neighbour(const GcPair& p, int x, int y, int dir, int& nx, int& ny) {
    nx = x + (dir == 0) - (dir == 1);
    ny = y + (dir == 2) - (dir == 3);
    return (unsigned)nx < (unsigned)p.W && (unsigned)ny < (unsigned)p.H;
}

// Capacities of one pair: the residual graph of the zero flow, and the excess of the saturated (reversed) source
// edges.
__global__ void __launch_bounds__(GC_BX * GC_BY) gc_caps_kernel(const __grid_constant__ GcPair p) {
    const int x = blockIdx.x * GC_BX + threadIdx.x, y = blockIdx.y * GC_BY + threadIdx.y;
    if (x >= p.W || y >= p.H) return;
    const long long u = (long long)y * p.W + x;
    bool s1, s2;
    int d;
    gc_pixel(p, x, y, s1, s2, d);
    p.e[u] = s2 && !s1 ? MCS_GC_TERMINAL : 0;
    p.rt[u] = s1 && !s2 ? MCS_GC_TERMINAL : 0;
#pragma unroll
    for (int dir = 0; dir < 4; ++dir) {
        int nx, ny, cap = 0;
        if (gc_neighbour(p, x, y, dir, nx, ny)) {
            bool t1, t2;
            int dn;
            gc_pixel(p, nx, ny, t1, t2, dn);
            cap = d + dn + 1 + (s1 && s2 && t1 && t2 ? 0 : MCS_GC_PENALTY);
        }
        p.r[dir * (long long)p.N + u] = cap;
    }
}

// Global relabel, first step: label 1 where the terminal edge has residual capacity, N elsewhere.
__global__ void __launch_bounds__(GC_BX * GC_BY) gc_label_init_kernel(const __grid_constant__ GcPair p) {
    const int x = blockIdx.x * GC_BX + threadIdx.x, y = blockIdx.y * GC_BY + threadIdx.y;
    if (x >= p.W || y >= p.H) return;
    const long long u = (long long)y * p.W + x;
    p.h[u] = p.rt[u] > 0 ? 1 : p.N;
}

// Global relabel, relaxation: h(u) = min(h(u), h(v) + 1) over the residual edges u -> v, inside a 32 x 32 tile until
// nothing changes (the halo holds the neighbours' labels at launch).  Labels only decrease toward the residual
// distances, so any interleaving converges to them; the host repeats the launch until a launch changes nothing.
__global__ void __launch_bounds__(GC_TILE * GC_BY) gc_relax_kernel(const __grid_constant__ GcPair p, int slot) {
    __shared__ int t[GC_TILE + 2][GC_TILE + 2];
    const int x0 = blockIdx.x * GC_TILE, y0 = blockIdx.y * GC_TILE;
    for (int i = threadIdx.y * GC_TILE + threadIdx.x; i < (GC_TILE + 2) * (GC_TILE + 2); i += GC_TILE * GC_BY) {
        const int tx = i % (GC_TILE + 2), ty = i / (GC_TILE + 2);
        const int x = x0 + tx - 1, y = y0 + ty - 1;
        t[ty][tx] = (unsigned)x < (unsigned)p.W && (unsigned)y < (unsigned)p.H ? p.h[(long long)y * p.W + x] : p.N;
    }
    constexpr int R = GC_TILE / GC_BY;
    int edges[R];   // bit dir: residual capacity toward that neighbour
    const int x = x0 + threadIdx.x;
#pragma unroll
    for (int k = 0; k < R; ++k) {
        const int y = y0 + threadIdx.y + k * GC_BY;
        edges[k] = 0;
        if (x < p.W && y < p.H) {
            const long long u = (long long)y * p.W + x;
#pragma unroll
            for (int dir = 0; dir < 4; ++dir)
                if (p.r[dir * (long long)p.N + u] > 0) edges[k] |= 1 << dir;
        }
    }
    __syncthreads();
    int any = 0;
    for (;;) {
        int changed = 0;
#pragma unroll
        for (int k = 0; k < R; ++k) {
            const int ty = threadIdx.y + k * GC_BY + 1, tx = threadIdx.x + 1;
            const int cur = t[ty][tx];
            int m = cur;
            if (edges[k] & 1) m = min(m, t[ty][tx + 1] + 1);
            if (edges[k] & 2) m = min(m, t[ty][tx - 1] + 1);
            if (edges[k] & 4) m = min(m, t[ty + 1][tx] + 1);
            if (edges[k] & 8) m = min(m, t[ty - 1][tx] + 1);
            if (m < cur) {
                t[ty][tx] = m;
                changed = 1;
            }
        }
        if (!__syncthreads_or(changed)) break;
        any = 1;
    }
    if (!any) return;
#pragma unroll
    for (int k = 0; k < R; ++k) {
        const int y = y0 + threadIdx.y + k * GC_BY;
        if (x < p.W && y < p.H) p.h[(long long)y * p.W + x] = t[threadIdx.y + k * GC_BY + 1][threadIdx.x + 1];
    }
    if (threadIdx.x == 0 && threadIdx.y == 0) atomicOr(p.flags + slot, 1);
}

// The active nodes: excess with a finite label.
__global__ void __launch_bounds__(GC_BX * GC_BY) gc_count_kernel(const __grid_constant__ GcPair p) {
    const int x = blockIdx.x * GC_BX + threadIdx.x, y = blockIdx.y * GC_BY + threadIdx.y;
    int active = 0;
    if (x < p.W && y < p.H) {
        const long long u = (long long)y * p.W + x;
        active = p.e[u] > 0 && p.h[u] < p.N;
    }
    active = __syncthreads_count(active);
    if (threadIdx.x == 0 && threadIdx.y == 0 && active) atomicAdd(p.flags + MCS_GC_RELAX, active);
}

// One round, first half: every active node pushes its excess to the terminal (label 0) and down the admissible
// edges (label one lower), touching only its own excess and residuals; out[] records what went each way.
__global__ void __launch_bounds__(GC_BX * GC_BY) gc_push_kernel(const __grid_constant__ GcPair p) {
    const int x = blockIdx.x * GC_BX + threadIdx.x, y = blockIdx.y * GC_BY + threadIdx.y;
    if (x >= p.W || y >= p.H) return;
    const long long u = (long long)y * p.W + x, N = p.N;
    int e = p.e[u];
    const int hu = p.h[u];
    int o[4] = {0, 0, 0, 0};
    if (e > 0 && hu < p.N) {
        if (hu == 1) {
            const int rt = p.rt[u];
            const int d = min(e, rt);
            if (d > 0) {
                p.rt[u] = rt - d;
                e -= d;
            }
        }
#pragma unroll
        for (int dir = 0; dir < 4; ++dir) {
            int nx, ny;
            if (e > 0 && gc_neighbour(p, x, y, dir, nx, ny)) {
                const int r = p.r[dir * N + u];
                if (r > 0 && p.h[(long long)ny * p.W + nx] == hu - 1) {
                    o[dir] = min(e, r);
                    p.r[dir * N + u] = r - o[dir];
                    e -= o[dir];
                }
            }
        }
        p.e[u] = e;
    }
#pragma unroll
    for (int dir = 0; dir < 4; ++dir) p.out[dir * N + u] = o[dir];
}

// One round, second half: take in what the neighbours pushed (excess, and residual back toward them), then relabel
// an active node without an admissible edge to one more than its lowest residual neighbour (labels of this round;
// the next round's go to h2).
__global__ void __launch_bounds__(GC_BX * GC_BY) gc_pull_kernel(const __grid_constant__ GcPair p) {
    const int x = blockIdx.x * GC_BX + threadIdx.x, y = blockIdx.y * GC_BY + threadIdx.y;
    if (x >= p.W || y >= p.H) return;
    const long long u = (long long)y * p.W + x, N = p.N;
    int e = p.e[u];
    int r[4], hv[4];
#pragma unroll
    for (int dir = 0; dir < 4; ++dir) {
        int nx, ny;
        r[dir] = p.r[dir * N + u];
        hv[dir] = p.N;
        if (gc_neighbour(p, x, y, dir, nx, ny)) {
            const long long v = (long long)ny * p.W + nx;
            const int in = p.out[(dir ^ 1) * N + v];   // right <-> left, down <-> up
            if (in) {
                e += in;
                r[dir] += in;
                p.r[dir * N + u] = r[dir];
            }
            hv[dir] = p.h[v];
        }
    }
    p.e[u] = e;
    const int hu = p.h[u];
    int hn = hu;
    if (e > 0 && hu < p.N) {
        const bool to_terminal = p.rt[u] > 0;
        bool admissible = to_terminal && hu == 1;
        int m = to_terminal ? 0 : p.N;
#pragma unroll
        for (int dir = 0; dir < 4; ++dir)
            if (r[dir] > 0) {
                admissible |= hv[dir] == hu - 1;
                m = min(m, hv[dir]);
            }
        if (!admissible) hn = min(p.N, m + 1);
    }
    p.h2[u] = hn;
}

// The cut inside the ROI: S = the pixels with a finite label after the last global relabel.
__global__ void __launch_bounds__(GC_BX * GC_BY) gc_cut_kernel(const __grid_constant__ GcPair p) {
    const int x = blockIdx.x * GC_BX + threadIdx.x + MCS_GC_GAP, y = blockIdx.y * GC_BY + threadIdx.y + MCS_GC_GAP;
    if (x >= p.W - MCS_GC_GAP || y >= p.H - MCS_GC_GAP) return;
    const bool in_s = p.h[(long long)y * p.W + x] < p.N;
    long long at[2];
    gc_inside(p, 0, x, y, at[0]);
    gc_inside(p, 1, x, y, at[1]);
    // inside the ROI both planes cover the pixel
    if (in_s && p.m[0][at[0]] != 0) p.m[1][at[1]] = 0;
    if (!in_s && p.m[1][at[1]] != 0) p.m[0][at[0]] = 0;
}

static dim3 gc_grid(int W, int H) { return dim3((W + GC_BX - 1) / GC_BX, (H + GC_BY - 1) / GC_BY, 1); }

// The global relabel of one pair; returns the active count (or -1 on a CUDA error, in e).
static long long gc_global_relabel(const GcPair& p, int* host, int& launches, cudaError_t& e) {
    const dim3 block(GC_BX, GC_BY, 1), tiles((p.W + GC_TILE - 1) / GC_TILE, (p.H + GC_TILE - 1) / GC_TILE, 1);
    gc_label_init_kernel<<<gc_grid(p.W, p.H), block>>>(p);
    ++launches;
    for (;;) {
        e = cudaMemsetAsync(p.flags, 0, (MCS_GC_RELAX + 1) * sizeof(int), 0);
        if (e != cudaSuccess) return -1;
        for (int s = 0; s < MCS_GC_RELAX; ++s) gc_relax_kernel<<<tiles, block>>>(p, s);
        gc_count_kernel<<<gc_grid(p.W, p.H), block>>>(p);
        launches += MCS_GC_RELAX + 1;
        e = cudaMemcpy(host, p.flags, (MCS_GC_RELAX + 1) * sizeof(int), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) return -1;
        if (host[MCS_GC_RELAX - 1] == 0) return host[MCS_GC_RELAX];
    }
}

// The sample table of every layer; returns the fed layers' count, their widest and tallest rectangle in bw, bh.
static int gc_sample_args(const mcs_plan* plan, const uint8_t* const* src, const int64_t* src_pitch, GcSample& a,
                          int& bw, int& bh) {
    memset(&a, 0, sizeof(a));
    int n = 0;
    bw = bh = 0;
    for (int k = 0; k < plan->n_layers; ++k) {
        const McsLayer& L = plan->layers[k];
        a.g[k] = L;
        a.src[k] = src[k];
        a.pitch[k] = src_pitch[k];
        const int x0 = L.rx0 > 0 ? L.rx0 : 0, y0 = L.ry0 > 0 ? L.ry0 : 0;
        const int x1 = L.rx1 < plan->out_w ? L.rx1 : plan->out_w, y1 = L.ry1 < plan->out_h ? L.ry1 : plan->out_h;
        a.rect[k] = make_int4(x0, y0, x1, y1);
        if (x1 > x0 && y1 > y0) {   // an empty rectangle feeds nothing
            a.layer[n++] = k;
            bw = x1 - x0 > bw ? x1 - x0 : bw;
            bh = y1 - y0 > bh ? y1 - y0 : bh;
        }
    }
    a.lut = plan->gains_on ? plan->d_gain_lut : nullptr;
    return n;
}

static void gc_sample_launch(const GcSample& a, int n, int bw, int bh) {
    const dim3 grid((bw + GC_BX - 1) / GC_BX, (bh + GC_BY - 1) / GC_BY, n), block(GC_BX, GC_BY, 1);
    if (a.lut)
        gc_sample_kernel<true><<<grid, block>>>(a);
    else
        gc_sample_kernel<false><<<grid, block>>>(a);
    mcs_count_launch(1);
}

int mcs_graphcut_sample(const mcs_plan* plan, const uint8_t* const* src, const int64_t* src_pitch, uint8_t* const* img,
                        bool gains, int* fed) {
    GcSample a;
    int bw, bh;
    const int n = gc_sample_args(plan, src, src_pitch, a, bw, bh);
    if (!gains) a.lut = nullptr;
    for (int u = 0; u < n; ++u) {
        fed[u] = a.layer[u];
        a.img[a.layer[u]] = img[a.layer[u]];
    }
    if (n > 0) gc_sample_launch(a, n, bw, bh);
    return n;
}

int mcs_graphcut_build(mcs_plan* plan, const uint8_t* const* src, const int64_t* src_pitch) {
    GcSample a;
    int bw, bh;
    const int n = gc_sample_args(plan, src, src_pitch, a, bw, bh);
    for (int u = 0; u < n; ++u)
        MCS_CHECK_ARG(src[a.layer[u]] != nullptr, "mcs_plan_set_graphcut_seams: src[%d] is NULL", a.layer[u]);
    int pi[MCS_MAX_LAYERS * MCS_MAX_LAYERS / 2], pj[MCS_MAX_LAYERS * MCS_MAX_LAYERS / 2];
    int np = 0;
    long long max_px = 0;
    for (int u = 0; u < n; ++u)
        for (int v = u + 1; v < n; ++v) {
            const int4 r1 = a.rect[a.layer[u]], r2 = a.rect[a.layer[v]];
            const int rx0 = max(r1.x, r2.x), ry0 = max(r1.y, r2.y), rx1 = min(r1.z, r2.z), ry1 = min(r1.w, r2.w);
            if (rx0 >= rx1 || ry0 >= ry1) continue;
            const long long px = (long long)(rx1 - rx0 + 2 * MCS_GC_GAP) * (ry1 - ry0 + 2 * MCS_GC_GAP);
            pi[np] = a.layer[u];
            pj[np] = a.layer[v];
            ++np;
            max_px = px > max_px ? px : max_px;
        }
    // everything goes to new planes; the plan changes only once every pair is cut
    uint8_t* planes[MCS_MAX_LAYERS] = {};
    int* scratch = nullptr;
    int* host = nullptr;
    cudaError_t e = cudaSuccess;
    int launches = 0, rc = MCS_OK;
    long long rounds = 0;
    for (int u = 0; u < n && e == cudaSuccess; ++u) {
        const int4 r = a.rect[a.layer[u]];
        e = cudaMalloc(&planes[a.layer[u]], (size_t)(r.z - r.x) * (r.w - r.y));
        if (e == cudaSuccess) e = cudaMalloc(&a.img[a.layer[u]], (size_t)(r.z - r.x) * (r.w - r.y) * 3);
    }
    if (e == cudaSuccess && np > 0) e = cudaMalloc(&scratch, ((size_t)12 * max_px + MCS_GC_RELAX + 1) * sizeof(int));
    if (e == cudaSuccess) e = cudaMallocHost(&host, (MCS_GC_RELAX + 1) * sizeof(int));
    if (e == cudaSuccess && n > 0) {
        mcs_seams_fill(plan, planes);
        gc_sample_launch(a, n, bw, bh);   // compensated when the plan has gains: the cut compares what is blended
        e = cudaGetLastError();
    }
    for (int q = 0; q < np && e == cudaSuccess && rc == MCS_OK; ++q) {
        GcPair p;
        const int i = pi[q], j = pj[q];
        const int4 r1 = a.rect[i], r2 = a.rect[j];
        const int rx0 = max(r1.x, r2.x), ry0 = max(r1.y, r2.y), rx1 = min(r1.z, r2.z), ry1 = min(r1.w, r2.w);
        p.W = rx1 - rx0 + 2 * MCS_GC_GAP;
        p.H = ry1 - ry0 + 2 * MCS_GC_GAP;
        p.N = p.W * p.H;
        const int4 rr[2] = {r1, r2};
        const int kk[2] = {i, j};
        for (int c = 0; c < 2; ++c) {
            p.m[c] = planes[kk[c]];
            p.img[c] = a.img[kk[c]];
            p.pw[c] = rr[c].z - rr[c].x;
            p.ph[c] = rr[c].w - rr[c].y;
            p.ox[c] = rx0 - MCS_GC_GAP - rr[c].x;
            p.oy[c] = ry0 - MCS_GC_GAP - rr[c].y;
        }
        p.e = scratch;
        p.h = scratch + max_px;
        p.h2 = scratch + 2 * max_px;
        p.rt = scratch + 3 * max_px;
        p.r = scratch + 4 * max_px;
        p.out = scratch + 8 * max_px;
        p.flags = scratch + 12 * max_px;
        const dim3 grid = gc_grid(p.W, p.H), block(GC_BX, GC_BY, 1);
        gc_caps_kernel<<<grid, block>>>(p);
        ++launches;
        for (;;) {
            const long long active = gc_global_relabel(p, host, launches, e);
            if (e != cudaSuccess || active == 0) break;
            if (rounds >= MCS_GC_MAX_ROUNDS) {
                mcs_set_error("mcs_plan_set_graphcut_seams: layers %d and %d: no maximum flow after %lld push-relabel "
                              "rounds (%lld nodes still active)", i, j, rounds, active);
                rc = MCS_ERR_CUDA;
                break;
            }
            for (int k = 0; k < MCS_GC_ROUNDS; ++k) {
                gc_push_kernel<<<grid, block>>>(p);
                gc_pull_kernel<<<grid, block>>>(p);
                int* t = p.h;
                p.h = p.h2;
                p.h2 = t;
            }
            launches += 2 * MCS_GC_ROUNDS;
            rounds += MCS_GC_ROUNDS;
        }
        if (e != cudaSuccess || rc != MCS_OK) break;
        gc_cut_kernel<<<gc_grid(rx1 - rx0, ry1 - ry0), block>>>(p);
        ++launches;
        e = cudaGetLastError();
    }
    mcs_count_launch(launches);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    if (scratch) cudaFree(scratch);
    if (host) cudaFreeHost(host);
    for (int k = 0; k < MCS_MAX_LAYERS; ++k)
        if (a.img[k]) cudaFree(a.img[k]);
    if (e != cudaSuccess && rc == MCS_OK) {
        mcs_set_error("mcs_plan_set_graphcut_seams: %s", cudaGetErrorString(e));
        rc = MCS_ERR_CUDA;
    }
    if (rc != MCS_OK) {
        for (int k = 0; k < MCS_MAX_LAYERS; ++k)
            if (planes[k]) cudaFree(planes[k]);
        return rc;
    }
    mcs_seams_free(plan);
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) plan->d_seam[k] = planes[k];
    plan->seams_on = 1;
    return MCS_OK;
}
