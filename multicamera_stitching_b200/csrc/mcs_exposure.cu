// Exposure compensation of the camera-weighted and multi-band blends (mcs_plan_estimate_gains,
// mcs_plan_set_exposure_gains, sm_100a): OpenCV's cv::detail::GainCompensator run on the cameras' overwrite samples
// v_k and weight samples w_k of one frame-set.  Specification: oracle/exposure_model.py.  Plan time only.
//
// Estimation, bit for bit with the specification:
//   1. seam_fill_kernel (mcs_seams.cu)          every fed layer's w_k over its clipped rectangle (the uncut weights)
//      gc_sample_kernel (mcs_seams_graphcut.cu) every fed layer's v_k, 3 bytes a pixel, never compensated
//   2. ex_stats_kernel, one launch, one warp per job, all jobs at once.  A job is one overlapping pair (i, j), i < j
//      in feed order, and one side of it (the image of i or of j), or one fed camera alone (i == j, counted only).
//      Over the overlap, row by row, each lane takes EX_PER_LANE pixels of a chunk: intersect = w_i == 255 &&
//      w_j == 255 is counted in integers, and the lane writes sqrt(double(b^2 + g^2 + r^2)) of an intersect pixel,
//      +0.0 elsewhere, to shared memory; lane 0 then adds the chunk in row-major order to its running sum.  Adding
//      +0.0 is exact, so the sum is the sequential sum over the intersect pixels that GainCompensator computes.
//   3. host: N = max(1, count), I = sum / N, the normal equations and their Gaussian elimination with partial
//      pivoting in plain float64 (the build has --fmad=false and -ffp-contract=off), operation for operation as
//      the specification states them.
// Apply: ex_lut_kernel writes one 256-entry table per layer, saturate_u8(rint(v * g)); the per-frame kernels of
// variants 5 and 6 and gc_sample_kernel look every camera's rounded sample up in it (their GAIN instantiations).
#include "mcs_device.cuh"

#include <math.h>
#include <string.h>

#define EX_ALPHA 0.01
#define EX_BETA 100.0
#define EX_PER_LANE 8
#define EX_CHUNK (32 * EX_PER_LANE)   // pixels of a row per step of a warp

struct ExJob {
    const uint8_t* m0;    // the two weight planes at the overlap's origin
    const uint8_t* m1;
    const uint8_t* img;   // the summed camera's samples at the overlap's origin (3 bytes a pixel), nullptr = count only
    int p0, p1, pimg;     // their row pitches in pixels (the planes' widths)
    int W, H;             // the overlap
};

__global__ void __launch_bounds__(32) ex_stats_kernel(const ExJob* __restrict__ jobs,
                                                      unsigned long long* __restrict__ count,
                                                      double* __restrict__ sum) {
    __shared__ double v[EX_CHUNK];
    const ExJob j = jobs[blockIdx.x];
    const int lane = threadIdx.x;
    unsigned long long c = 0;
    double s = 0.0;   // lane 0's running sum
    for (int y = 0; y < j.H; ++y) {
        const uint8_t* r0 = j.m0 + (long long)y * j.p0;
        const uint8_t* r1 = j.m1 + (long long)y * j.p1;
        const uint8_t* ri = j.img ? j.img + (long long)y * j.pimg * 3 : nullptr;
        for (int x0 = 0; x0 < j.W; x0 += EX_CHUNK) {
#pragma unroll
            for (int t = 0; t < EX_PER_LANE; ++t) {
                const int x = x0 + t * 32 + lane;
                const bool in = x < j.W && __ldg(r0 + x) == 255 && __ldg(r1 + x) == 255;
                c += in ? 1 : 0;
                double n = 0.0;
                if (in && ri) {
                    const int b = __ldg(ri + 3 * x), g = __ldg(ri + 3 * x + 1), r = __ldg(ri + 3 * x + 2);
                    n = __dsqrt_rn((double)(b * b + g * g + r * r));
                }
                v[t * 32 + lane] = n;
            }
            __syncwarp();
            if (ri && lane == 0) {
                const int m = j.W - x0 < EX_CHUNK ? j.W - x0 : EX_CHUNK;
                for (int k = 0; k < m; ++k) s = __dadd_rn(s, v[k]);
            }
            __syncwarp();
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
    if (lane == 0) {
        count[blockIdx.x] = c;
        sum[blockIdx.x] = s;
    }
}

struct ExLut {
    double g[MCS_MAX_LAYERS];
};

// One block per layer: table[v] = saturate_u8(rint(v * g)), rounding half to even as cvRound does.
__global__ void __launch_bounds__(256) ex_lut_kernel(const __grid_constant__ ExLut a, uint8_t* __restrict__ lut) {
    const int k = blockIdx.x, v = threadIdx.x;
    const int r = __double2int_rn(__dmul_rn((double)v, a.g[k]));   // saturates to the int range
    lut[k * 256 + v] = (uint8_t)(r < 0 ? 0 : r > 255 ? 255 : r);
}

void mcs_exposure_free(mcs_plan* plan) {
    if (plan->d_gain_lut) cudaFree(plan->d_gain_lut);
    plan->d_gain_lut = nullptr;
    plan->gains_on = 0;
}

// The gains of the n cameras not skipped, from N and I (n_all x n_all, row-major) by the normal equations of
// GainCompensator and Gaussian elimination with partial pivoting.  A is symmetric positive definite (its diagonal
// holds beta * N(i, i) >= 100), so no pivot vanishes.
static void ex_solve(int n_all, const long long* N, const double* I, const bool* skip, double* gains) {
    int cams[MCS_MAX_LAYERS];
    int m = 0;
    for (int i = 0; i < n_all; ++i) {
        gains[i] = 1.0;
        if (!skip[i]) cams[m++] = i;
    }
    if (m == 0) return;
    double A[MCS_MAX_LAYERS][MCS_MAX_LAYERS] = {};
    double b[MCS_MAX_LAYERS] = {};
    for (int ki = 0; ki < m; ++ki)
        for (int kj = 0; kj < m; ++kj) {
            const int i = cams[ki], j = cams[kj];
            const double nij = (double)N[i * n_all + j], iij = I[i * n_all + j], iji = I[j * n_all + i];
            b[ki] += EX_BETA * nij;
            A[ki][ki] += EX_BETA * nij;
            if (j != i) {
                A[ki][ki] += 2 * EX_ALPHA * iij * iij * nij;
                A[ki][kj] -= 2 * EX_ALPHA * iij * iji * nij;
            }
        }
    for (int i = 0; i < m; ++i) {
        int k = i;
        for (int j = i + 1; j < m; ++j)
            if (fabs(A[j][i]) > fabs(A[k][i])) k = j;
        if (k != i) {
            for (int j = i; j < m; ++j) {
                const double t = A[i][j];
                A[i][j] = A[k][j];
                A[k][j] = t;
            }
            const double t = b[i];
            b[i] = b[k];
            b[k] = t;
        }
        const double d = -1.0 / A[i][i];
        for (int j = i + 1; j < m; ++j) {
            const double alpha = A[j][i] * d;
            for (int c = i + 1; c < m; ++c) A[j][c] += alpha * A[i][c];
            b[j] += alpha * b[i];
        }
    }
    for (int i = m - 1; i >= 0; --i) {
        double s = b[i];
        for (int c = i + 1; c < m; ++c) s -= A[i][c] * b[c];
        b[i] = s / A[i][i];
    }
    for (int k = 0; k < m; ++k) gains[cams[k]] = b[k];
}

extern "C" int mcs_plan_estimate_gains(const mcs_plan* plan, const uint8_t* const* src, const int64_t* src_pitch,
                                       double* host_gains, int64_t* host_N, double* host_I) {
    MCS_CHECK_ARG(plan != nullptr && src != nullptr && src_pitch != nullptr && host_gains != nullptr,
                  "mcs_plan_estimate_gains: NULL argument");
    MCS_CHECK_ARG(plan->cw_maps, "mcs_plan_estimate_gains: the plan has no camera weights (mcs_plan_set_camera_weights)");
    if (plan->channels != 3) {
        mcs_set_error("mcs_plan_estimate_gains: GainCompensator estimates on 3 channels, the plan has %d",
                      plan->channels);
        return MCS_ERR_UNSUPPORTED;
    }
    int4 rect[MCS_MAX_LAYERS];
    int fed[MCS_MAX_LAYERS];
    int n = 0;
    for (int k = 0; k < plan->n_layers; ++k) {
        const McsLayer& L = plan->layers[k];
        const int x0 = L.rx0 > 0 ? L.rx0 : 0, y0 = L.ry0 > 0 ? L.ry0 : 0;
        const int x1 = L.rx1 < plan->out_w ? L.rx1 : plan->out_w, y1 = L.ry1 < plan->out_h ? L.ry1 : plan->out_h;
        rect[k] = make_int4(x0, y0, x1, y1);
        if (x1 > x0 && y1 > y0) {   // an empty rectangle feeds nothing
            MCS_CHECK_ARG(src[k] != nullptr, "mcs_plan_estimate_gains: src[%d] is NULL", k);
            fed[n++] = k;
        }
    }
    uint8_t* planes[MCS_MAX_LAYERS] = {};
    uint8_t* imgs[MCS_MAX_LAYERS] = {};
    cudaError_t e = cudaSuccess;
    for (int u = 0; u < n && e == cudaSuccess; ++u) {
        const int4 r = rect[fed[u]];
        e = cudaMalloc(&planes[fed[u]], (size_t)(r.z - r.x) * (r.w - r.y));
        if (e == cudaSuccess) e = cudaMalloc(&imgs[fed[u]], (size_t)(r.z - r.x) * (r.w - r.y) * 3);
    }
    // jobs: every fed camera alone (its N(i, i)), then both sides of every overlapping pair; job q sums the image of
    // fed camera ju[q] over its overlap with jv[q]
    constexpr int MAX_JOBS = MCS_MAX_LAYERS * MCS_MAX_LAYERS;
    ExJob jobs[MAX_JOBS];
    int ju[MAX_JOBS], jv[MAX_JOBS];
    int nj = 0;
    for (int u = 0; u < n; ++u)
        for (int v = u; v < n; ++v) {
            const int a = fed[u], c = fed[v];
            const int4 r1 = rect[a], r2 = rect[c];
            const int rx0 = max(r1.x, r2.x), ry0 = max(r1.y, r2.y), rx1 = min(r1.z, r2.z), ry1 = min(r1.w, r2.w);
            if (rx0 >= rx1 || ry0 >= ry1) continue;
            const long long o1 = (long long)(ry0 - r1.y) * (r1.z - r1.x) + (rx0 - r1.x);
            const long long o2 = (long long)(ry0 - r2.y) * (r2.z - r2.x) + (rx0 - r2.x);
            for (int side = 0; side < (u == v ? 1 : 2); ++side) {
                ExJob& J = jobs[nj];
                J.m0 = planes[a] + o1;
                J.m1 = planes[c] + o2;
                J.p0 = r1.z - r1.x;
                J.p1 = r2.z - r2.x;
                J.img = u == v ? nullptr : side == 0 ? imgs[a] + 3 * o1 : imgs[c] + 3 * o2;
                J.pimg = side == 0 ? J.p0 : J.p1;
                J.W = rx1 - rx0;
                J.H = ry1 - ry0;
                ju[nj] = side == 0 ? u : v;
                jv[nj] = side == 0 ? v : u;
                ++nj;
            }
        }
    ExJob* d_jobs = nullptr;
    unsigned long long* d_count = nullptr;
    unsigned long long h_count[MAX_JOBS];
    double h_sum[MAX_JOBS];
    if (e == cudaSuccess && nj > 0) e = cudaMalloc(&d_jobs, sizeof(ExJob) * nj);
    if (e == cudaSuccess && nj > 0) e = cudaMalloc(&d_count, (sizeof(unsigned long long) + sizeof(double)) * nj);
    if (e == cudaSuccess && nj > 0) {
        double* d_sum = reinterpret_cast<double*>(d_count + nj);
        e = cudaMemcpy(d_jobs, jobs, sizeof(ExJob) * nj, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) {
            int order[MCS_MAX_LAYERS];
            mcs_seams_fill(plan, planes);
            mcs_graphcut_sample(plan, src, src_pitch, imgs, false, order);
            ex_stats_kernel<<<nj, 32>>>(d_jobs, d_count, d_sum);
            mcs_count_launch(1);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpy(h_count, d_count, sizeof(unsigned long long) * nj, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(h_sum, d_sum, sizeof(double) * nj, cudaMemcpyDeviceToHost);
    }
    if (d_jobs) cudaFree(d_jobs);
    if (d_count) cudaFree(d_count);
    for (int k = 0; k < MCS_MAX_LAYERS; ++k) {
        if (planes[k]) cudaFree(planes[k]);
        if (imgs[k]) cudaFree(imgs[k]);
    }
    if (e != cudaSuccess) {
        mcs_set_error("mcs_plan_estimate_gains: %s", cudaGetErrorString(e));
        return MCS_ERR_CUDA;
    }
    long long N[MCS_MAX_LAYERS * MCS_MAX_LAYERS] = {};
    double I[MCS_MAX_LAYERS * MCS_MAX_LAYERS] = {};
    bool skip[MCS_MAX_LAYERS];
    for (int u = 0; u < n; ++u) skip[u] = true;
    for (int q = 0; q < nj; ++q) {
        const int i = ju[q], j = jv[q];
        const long long c = (long long)h_count[q];
        N[i * n + j] = N[j * n + i] = c > 1 ? c : 1;
        if (i == j || c == 0) continue;
        skip[i] = skip[j] = false;
        I[i * n + j] = h_sum[q] / (double)N[i * n + j];
    }
    double g[MCS_MAX_LAYERS];
    ex_solve(n, N, I, skip, g);
    for (int k = 0; k < plan->n_layers; ++k) host_gains[k] = 1.0;   // a layer that feeds nothing
    for (int u = 0; u < n; ++u) host_gains[fed[u]] = g[u];
    for (int q = 0; q < n * n; ++q) {
        if (host_N) host_N[q] = N[q];
        if (host_I) host_I[q] = I[q];
    }
    return MCS_OK;
}

extern "C" int mcs_plan_set_exposure_gains(mcs_plan* plan, const double* gains) {
    MCS_CHECK_ARG(plan != nullptr, "mcs_plan_set_exposure_gains: plan is NULL");
    MCS_CHECK_ARG(plan->cw_maps, "mcs_plan_set_exposure_gains: the plan has no camera weights (mcs_plan_set_camera_weights)");
    if (gains == nullptr) {
        mcs_exposure_free(plan);
        return MCS_OK;
    }
    ExLut a;
    memset(&a, 0, sizeof(a));
    for (int k = 0; k < plan->n_layers; ++k) {
        MCS_CHECK_ARG(isfinite(gains[k]) && gains[k] >= 0.0, "mcs_plan_set_exposure_gains: gain %d is %g (finite and "
                      ">= 0 needed)", k, gains[k]);
        a.g[k] = gains[k];
    }
    if (!plan->d_gain_lut) MCS_CHECK_CUDA(cudaMalloc(&plan->d_gain_lut, MCS_MAX_LAYERS * 256));
    ex_lut_kernel<<<plan->n_layers, 256>>>(a, plan->d_gain_lut);
    mcs_count_launch(1);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) {
        mcs_exposure_free(plan);
        mcs_set_error("mcs_plan_set_exposure_gains: %s", cudaGetErrorString(e));
        return MCS_ERR_CUDA;
    }
    plan->gains_on = 1;
    return MCS_OK;
}
