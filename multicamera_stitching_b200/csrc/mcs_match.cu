// Brute-force Hamming 2-NN + ratio test (sm_100a): XOR + POPC on the integer pipe, per-lane
// running top-2, warp-shuffle merge.  Replaces cv2 BFMatcher.knnMatch(k=2) + the ratio loop of
// StitcherBase.matchKeypoints (StitcherClass.py:423-433) for binary descriptors.
//
// Layout: one CTA stages a chunk of the train set in shared memory *word-transposed*
// (word w of descriptor j at [w][j]) so that the 32 lanes of a warp, each owning one train
// descriptor, read consecutive banks.  Each warp owns one query at a time; the query words sit
// in registers.  A candidate is ordered by the packed key (distance << 21 | train index), which
// gives cv2's tie-break (lower train index first) for free.
#include "mcs_common.h"

#define MATCH_THREADS 256
#define MATCH_WARPS (MATCH_THREADS / 32)
#define MATCH_CHUNK 2048            // train descriptors per shared-memory pass
#define MATCH_IDX_BITS 21
#define MATCH_KEY_NONE 0xFFFFFFFFu

__device__ __forceinline__ void top2_insert(uint32_t key, uint32_t& k0, uint32_t& k1) {
    const uint32_t hi = max(k0, key);
    k0 = min(k0, key);
    k1 = min(k1, hi);
}

template <int WORDS>
__global__ void __launch_bounds__(MATCH_THREADS)
mcs_match_top2_kernel(const uint8_t* __restrict__ q, const int32_t* __restrict__ nq_arr, int nq_max,
                      const uint8_t* __restrict__ t, const int32_t* __restrict__ nt_arr, int nt_max,
                      double ratio, int32_t* __restrict__ idx2, int32_t* __restrict__ dist2,
                      uint8_t* __restrict__ keep, int queries_per_cta) {
    extern __shared__ uint32_t s_train[];  // [WORDS][MATCH_CHUNK]
    const int pair = blockIdx.y;
    const int nq = nq_arr ? min(nq_arr[pair], nq_max) : nq_max;
    const int nt = nt_arr ? min(nt_arr[pair], nt_max) : nt_max;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q_begin = blockIdx.x * queries_per_cta;
    const int q_end = min(q_begin + queries_per_cta, nq_max);
    if (q_begin >= nq_max) return;

    const uint32_t* tw = reinterpret_cast<const uint32_t*>(t + (size_t)pair * nt_max * (WORDS * 4));
    const uint32_t* qw = reinterpret_cast<const uint32_t*>(q + (size_t)pair * nq_max * (WORDS * 4));

    // Running best / second best of every query this warp owns across train chunks.  A warp
    // owns queries q_begin + warp, + MATCH_WARPS, ... ; at most 4 per warp are kept in
    // registers per sweep (queries_per_cta <= 4 * MATCH_WARPS).
    constexpr int QPW = 4;
    uint32_t best0[QPW], best1[QPW];
#pragma unroll
    for (int i = 0; i < QPW; ++i) best0[i] = best1[i] = MATCH_KEY_NONE;

    for (int c0 = 0; c0 < nt; c0 += MATCH_CHUNK) {
        const int cn = min(MATCH_CHUNK, nt - c0);
        __syncthreads();
        // stage: coalesced 32-bit reads, transposed writes
        for (int i = threadIdx.x; i < cn * WORDS; i += MATCH_THREADS) {
            const int j = i / WORDS, w = i - j * WORDS;
            s_train[w * MATCH_CHUNK + j] = __ldg(tw + (size_t)(c0 + j) * WORDS + w);
        }
        __syncthreads();
#pragma unroll
        for (int qi = 0; qi < QPW; ++qi) {
            const int qidx = q_begin + warp + qi * MATCH_WARPS;
            if (qidx >= q_end || qidx >= nq) continue;  // warp-uniform
            uint32_t qr[WORDS];
#pragma unroll
            for (int w = 0; w < WORDS; ++w) qr[w] = __ldg(qw + (size_t)qidx * WORDS + w);
            uint32_t k0 = best0[qi], k1 = best1[qi];
            for (int j = lane; j < cn; j += 32) {
                uint32_t d = 0;
#pragma unroll
                for (int w = 0; w < WORDS; ++w) d += __popc(qr[w] ^ s_train[w * MATCH_CHUNK + j]);
                top2_insert((d << MATCH_IDX_BITS) | (uint32_t)(c0 + j), k0, k1);
            }
            best0[qi] = k0;
            best1[qi] = k1;
        }
    }

    // merge the 32 per-lane (best, second) pairs of each query and emit
#pragma unroll
    for (int qi = 0; qi < QPW; ++qi) {
        const int qidx = q_begin + warp + qi * MATCH_WARPS;
        if (qidx >= q_end) continue;
        uint32_t k0 = best0[qi], k1 = best1[qi];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const uint32_t o0 = __shfl_xor_sync(0xffffffffu, k0, off);
            const uint32_t o1 = __shfl_xor_sync(0xffffffffu, k1, off);
            const uint32_t lo = min(k0, o0), hi = max(k0, o0);
            k1 = min(hi, min(k1, o1));
            k0 = lo;
        }
        if (lane == 0) {
            const size_t o = (size_t)pair * nq_max + qidx;
            const bool valid_q = qidx < nq;
            const bool h0 = valid_q && k0 != MATCH_KEY_NONE, h1 = valid_q && k1 != MATCH_KEY_NONE;
            const int d0 = (int)(k0 >> MATCH_IDX_BITS), d1 = (int)(k1 >> MATCH_IDX_BITS);
            idx2[2 * o] = h0 ? (int)(k0 & ((1u << MATCH_IDX_BITS) - 1)) : -1;
            idx2[2 * o + 1] = h1 ? (int)(k1 & ((1u << MATCH_IDX_BITS) - 1)) : -1;
            dist2[2 * o] = h0 ? d0 : -1;
            dist2[2 * o + 1] = h1 ? d1 : -1;
            // `m[0].distance < m[1].distance * ratio` in Python floats (float64)
            keep[o] = (h0 && h1 && (double)d0 < __dmul_rn((double)d1, ratio)) ? 1 : 0;
        }
    }
}

template <int WORDS>
static cudaError_t launch_match(const uint8_t* q, const int32_t* nq, int nq_max, const uint8_t* t,
                                const int32_t* nt, int nt_max, double ratio, int32_t* idx2,
                                int32_t* dist2, uint8_t* keep, int batch, cudaStream_t stream) {
    const size_t smem = (size_t)WORDS * MATCH_CHUNK * sizeof(uint32_t);
    cudaError_t e = cudaFuncSetAttribute(mcs_match_top2_kernel<WORDS>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    // Enough CTAs to cover the 148 SMs a few times over while amortising the train staging.
    int qpc = 4 * MATCH_WARPS;
    while (qpc > MATCH_WARPS && (long long)((nq_max + qpc - 1) / qpc) * batch < 2 * 148) qpc -= MATCH_WARPS;
    dim3 grid((nq_max + qpc - 1) / qpc, batch, 1);
    mcs_match_top2_kernel<WORDS><<<grid, MATCH_THREADS, smem, stream>>>(q, nq, nq_max, t, nt, nt_max, ratio,
                                                                       idx2, dist2, keep, qpc);
    mcs_count_launch(1);
    return cudaGetLastError();
}

extern "C" int mcs_match_hamming_top2(const uint8_t* q, const int32_t* nq, int nq_max,
                                      const uint8_t* t, const int32_t* nt, int nt_max,
                                      int desc_bytes, double ratio, int32_t* idx2, int32_t* dist2,
                                      uint8_t* keep, int batch, void* cuda_stream) {
    MCS_CHECK_ARG(batch >= 0 && batch <= 65535, "mcs_match_hamming_top2: batch=%d outside 0..65535", batch);
    MCS_CHECK_ARG(nq_max >= 0 && nt_max >= 0 && nt_max < (1 << MATCH_IDX_BITS),
                  "mcs_match_hamming_top2: nq_max=%d nt_max=%d out of range", nq_max, nt_max);
    MCS_CHECK_ARG(desc_bytes == 32 || desc_bytes == 64 || desc_bytes == 16,
                  "mcs_match_hamming_top2: desc_bytes=%d (supported: 16, 32, 64)", desc_bytes);
    if (batch == 0 || nq_max == 0) return MCS_OK;
    MCS_CHECK_ARG(q && idx2 && dist2 && keep && (t || nt_max == 0), "mcs_match_hamming_top2: NULL buffer");
    MCS_CHECK_ARG(((uintptr_t)q & 3) == 0 && ((uintptr_t)t & 3) == 0,
                  "mcs_match_hamming_top2: descriptor buffers must be 4-byte aligned");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    cudaError_t e;
    if (desc_bytes == 32)
        e = launch_match<8>(q, nq, nq_max, t, nt, nt_max, ratio, idx2, dist2, keep, batch, stream);
    else if (desc_bytes == 64)
        e = launch_match<16>(q, nq, nq_max, t, nt, nt_max, ratio, idx2, dist2, keep, batch, stream);
    else
        e = launch_match<4>(q, nq, nq_max, t, nt, nt_max, ratio, idx2, dist2, keep, batch, stream);
    if (e != cudaSuccess) {
        mcs_set_error("mcs_match_hamming_top2: launch failed: %s", cudaGetErrorString(e));
        return MCS_ERR_CUDA;
    }
    return MCS_OK;
}

// -------------------------------------------------------------------------------------------------
// Brute-force L2 2-NN + ratio test for float32 descriptors: the reference's own matcher branch
// (SIFT, 128 floats, cv2.DescriptorMatcher_create("BruteForce") = NORM_L2, StitcherClass.py:380-386,
// :423-433).
//
// distance = sqrtf(sum_k (a_k - b_k)^2), the difference form OpenCV's normL2Sqr uses (no
// |a|^2 + |b|^2 - 2ab expansion: that form cancels).  SIFT descriptors as OpenCV emits them are
// integer-valued floats in 0..255, so every square and every partial sum (< 128 * 255^2 < 2^24) is exact
// in float32 whatever the order of summation: distances, neighbour order and ratio decisions are then
// bit-identical to cv2's.  For other float descriptors the sum is rounded in this kernel's order
// (k ascending, one accumulator), which may differ from OpenCV's SIMD order in the last bit.
//
// No tensor cores: the work is 2000 x 2000 x 128 x 4 pairs = 2 GFLOP of FP32 multiply-adds, tens of
// microseconds on the FMA pipe next to a second of CPU SIFT detection per frame, and an MMA would need
// the cancelling expansion above.
//
// Layout: a CTA owns 32 queries and sweeps the train set in chunks of 128; both tiles sit in shared memory
// with a row pitch of DIM + 1 floats (conflict-free column walks).  Thread (ty, lane) accumulates the 4 x 4
// distances between queries 4 ty .. 4 ty + 3 and trains lane, lane + 32, lane + 64, lane + 96 of the chunk,
// keeps a running top-2 per query (packed key: sqrtf(sum) bits << 32 | train index, which orders
// non-negative floats numerically and breaks ties toward the lower index), and the 32 lanes merge by
// shuffles at the end.
#define L2_QB 32
#define L2_TB 128
#define L2_THREADS 256

__device__ __forceinline__ void top2_insert64(unsigned long long key, unsigned long long& k0, unsigned long long& k1) {
    const unsigned long long hi = k0 > key ? k0 : key;
    k0 = k0 < key ? k0 : key;
    k1 = k1 < hi ? k1 : hi;
}

__global__ void __launch_bounds__(L2_THREADS)
mcs_match_l2_kernel(const float* __restrict__ q, const int32_t* __restrict__ nq_arr, int nq_max,
                    const float* __restrict__ t, const int32_t* __restrict__ nt_arr, int nt_max, int dim,
                    double ratio, int32_t* __restrict__ idx2, float* __restrict__ dist2, uint8_t* __restrict__ keep) {
    extern __shared__ float s_l2[];
    const int pitch = dim + 1;
    float* s_q = s_l2;                    // [L2_QB][pitch]
    float* s_t = s_l2 + L2_QB * pitch;    // [L2_TB][pitch]
    const int pair = blockIdx.y;
    const int nq = nq_arr ? min(nq_arr[pair], nq_max) : nq_max;
    const int nt = nt_arr ? min(nt_arr[pair], nt_max) : nt_max;
    const int q0 = blockIdx.x * L2_QB;
    if (q0 >= nq_max) return;
    const int ty = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* qp = q + (size_t)pair * nq_max * dim;
    const float* tp = t + (size_t)pair * nt_max * dim;

    for (int i = threadIdx.x; i < L2_QB * dim; i += L2_THREADS) {
        const int r = i / dim, k = i - r * dim;
        s_q[r * pitch + k] = q0 + r < nq ? __ldg(qp + (size_t)(q0 + r) * dim + k) : 0.0f;
    }
    const unsigned long long none = ~0ull;
    unsigned long long b0[4], b1[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) b0[i] = b1[i] = none;

    for (int c0 = 0; c0 < nt; c0 += L2_TB) {
        const int cn = min(L2_TB, nt - c0);
        __syncthreads();
        for (int i = threadIdx.x; i < L2_TB * dim; i += L2_THREADS) {
            const int r = i / dim, k = i - r * dim;
            s_t[r * pitch + k] = r < cn ? __ldg(tp + (size_t)(c0 + r) * dim + k) : 0.0f;
        }
        __syncthreads();
        float acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = 0.0f;
        for (int k = 0; k < dim; ++k) {
            float qa[4], tb[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) qa[a] = s_q[(4 * ty + a) * pitch + k];
#pragma unroll
            for (int b = 0; b < 4; ++b) tb[b] = s_t[(lane + 32 * b) * pitch + k];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const float d = __fsub_rn(qa[a], tb[b]);
                    acc[a][b] = __fadd_rn(acc[a][b], __fmul_rn(d, d));   // like the reference build: no contraction
                }
        }
        // Rank by the rooted distance, as cv2's batchDistance does: sqrtf maps neighbouring sums to one float
        // (e.g. 4200782 and 4200783), and among equal distances the lower train index must win, whichever
        // sum was smaller.
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int j = lane + 32 * b;
                if (j < cn)
                    top2_insert64(((unsigned long long)__float_as_uint(sqrtf(acc[a][b])) << 32) | (unsigned)(c0 + j),
                                  b0[a], b1[a]);
            }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        unsigned long long k0 = b0[a], k1 = b1[a];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const unsigned long long o0 = __shfl_xor_sync(0xffffffffu, k0, off);
            const unsigned long long o1 = __shfl_xor_sync(0xffffffffu, k1, off);
            const unsigned long long lo = k0 < o0 ? k0 : o0, hi = k0 < o0 ? o0 : k0;
            const unsigned long long m1 = k1 < o1 ? k1 : o1;
            k1 = hi < m1 ? hi : m1;
            k0 = lo;
        }
        const int qidx = q0 + 4 * ty + a;
        if (lane == 0 && qidx < nq_max) {
            const size_t o = (size_t)pair * nq_max + qidx;
            const bool valid_q = qidx < nq;
            const bool h0 = valid_q && k0 != none, h1 = valid_q && k1 != none;
            const float d0 = __uint_as_float((unsigned)(k0 >> 32)), d1 = __uint_as_float((unsigned)(k1 >> 32));
            idx2[2 * o] = h0 ? (int)(unsigned)k0 : -1;
            idx2[2 * o + 1] = h1 ? (int)(unsigned)k1 : -1;
            dist2[2 * o] = h0 ? d0 : -1.0f;
            dist2[2 * o + 1] = h1 ? d1 : -1.0f;
            // `m[0].distance < m[1].distance * ratio`: float32 distances promoted to Python floats
            keep[o] = (h0 && h1 && (double)d0 < __dmul_rn((double)d1, ratio)) ? 1 : 0;
        }
    }
}

extern "C" int mcs_match_l2_top2(const float* q, const int32_t* nq, int nq_max, const float* t, const int32_t* nt,
                                 int nt_max, int dim, double ratio, int32_t* idx2, float* dist2, uint8_t* keep,
                                 int batch, void* cuda_stream) {
    MCS_CHECK_ARG(batch >= 0 && batch <= 65535, "mcs_match_l2_top2: batch=%d outside 0..65535", batch);
    MCS_CHECK_ARG(nq_max >= 0 && nt_max >= 0, "mcs_match_l2_top2: nq_max=%d nt_max=%d out of range", nq_max, nt_max);
    MCS_CHECK_ARG(dim >= 1 && dim <= 256, "mcs_match_l2_top2: dim=%d outside 1..256", dim);
    if (batch == 0 || nq_max == 0) return MCS_OK;
    MCS_CHECK_ARG(q && idx2 && dist2 && keep && (t || nt_max == 0), "mcs_match_l2_top2: NULL buffer");
    const size_t smem = (size_t)(L2_QB + L2_TB) * (dim + 1) * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(mcs_match_l2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
        dim3 grid((nq_max + L2_QB - 1) / L2_QB, batch, 1);
        mcs_match_l2_kernel<<<grid, L2_THREADS, smem, (cudaStream_t)cuda_stream>>>(q, nq, nq_max, t, nt, nt_max, dim, ratio,
                                                                                   idx2, dist2, keep);
        mcs_count_launch(1);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) {
        mcs_set_error("mcs_match_l2_top2: launch failed: %s", cudaGetErrorString(e));
        return MCS_ERR_CUDA;
    }
    return MCS_OK;
}
