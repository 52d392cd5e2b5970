// Variant 2 ("tiled") of the fused warp + paste kernel (sm_100a).
//
// Persistent CTAs (two per SM) of eight resampling warps and one producer warpgroup walk the plan's
// tile table.  A work unit is one 128 x 16 output cell of one layer for one frame; a CHUNK is a run
// of consecutive frames of one cell.
//
//   staging   The bounding box of the source pixels a WARP / COPY cell touches is brought into a
//             ring of shared-memory buffers by the TMA engine (cp.async.bulk.tensor.3d, zero fill
//             outside the image = cv2's BORDER_CONSTANT 0), one box per unit.  One thread of the
//             producer warpgroup claims the chunks, copies their records and issues every box as
//             soon as all resampling warps have released its slot (full / empty mbarriers per slot,
//             no CTA-wide barrier anywhere in the loop), so the ring is kept full whatever warp is
//             behind.  The producer warpgroup gives its registers to the resampling warps
//             (setmaxnreg): 32 a thread against 104, which keeps two CTAs per SM.
//   resample  warp w owns cell rows w and w + 8, lane l the columns l, l+32, l+64, l+96
//             (consecutive lanes read consecutive source pixels: bank-conflict free).
//
// Everything OpenCV's coordinate recipe produces - the float64 projective division, the 1/32-px
// rounding, tap clamping - is frame- AND launch-invariant, so it is evaluated once, at plan time
// (mcs_tiles.cu), into one 32-bit descriptor per output pixel: byte offset of the tap window
// inside the staged box, ax, ay.  A chunk starts by expanding its thread's 8 descriptors into
// registers (window address, byte phase, four 16-bit tap weights 64*wy*wx); the hot loop is
// integer only.  Per frame a pixel costs six aligned LDS.32, two funnel shifts and two byte
// permutes per source row, two IDP.2A per channel, and a 16-bit + a byte store into the warp's
// private rows of the output staging area, which the same warp streams to the panorama with
// 16-byte stores (the staging rows are pre-shifted to the destination's 16-byte phase, so that
// copy is LDS.128 -> STG.128 without realignment).
//
// Work split (see mcs_launch_tiled): frames are processed in blocks of a few frames; inside a
// block the CTAs sweep the tile table class by class, whole cells round-robin and the leftover
// cells cut into equal-cost runs, so that at any time all CTAs work side by side on neighbouring
// cells of the same few frames.
// Every source byte is fetched once per cell that touches it, every output byte is written once.
#include "mcs_device.cuh"

#include <cuda.h>   // CUtensorMap
#include <string.h>
#include <stdlib.h>

#define TILED_WARPS MCS_TILED_WARPS
#define TILED_THREADS (32 * TILED_WARPS)            // resampling threads; the producer warpgroup follows them
#define TILED_CTA_THREADS (TILED_THREADS + 128)
#define TILED_MIN_CTAS 2
// setmaxnreg moves registers inside one CTA's pool, which is fixed at launch: 384 threads x 80 registers (two
// CTAs per SM).  128 x 32 + 256 x 104 fills it exactly; the resampling loops need no spill at 104.
#define TILED_PRODUCER_REGS 32
#define TILED_CONSUMER_REGS 104
#define TILED_PX_BATCH 4   // pixels whose loads are issued before the first store
#define TILED_SMEM_BUDGET_KB 113   // per CTA, so that TILED_MIN_CTAS CTAs fit an SM
#define TILED_MAX_STAGES 8

struct TiledArgs {
    CUtensorMap tmap[MCS_MAX_LAYERS];   // source of each layer as (row words, rows, frames) of uint32
    const McsTile* tiles;
    const int4* issue;                  // per tile {layer, bx, by, box bytes}: all the producer needs of a tile
    const McsLayer* layers;
    const uint32_t* desc;               // plan-time pixel descriptors, 2048 per WARP tile
    uint8_t* dst;
    long long dst_pitch;
    long long dst_frame_stride;
    int box_bytes;                      // bytes of one staging buffer
    int stages;                         // staging buffers in the ring (3..TILED_MAX_STAGES)
    // Work split.  A CHUNK is one tile (cell) for the frames of one frame block; chunk id = block * n_tiles +
    // tile, i.e. the tile table (sorted FAST, WARP, COPY, ZERO) is swept once per frame block.  The CTAs
    // claim chunks at run time, `claim` consecutive ids per atomic on work[0]: whoever is served faster by
    // the memory system simply takes more of them (a static split left the slowest CTA 5 % behind the
    // median with resampling and 13 % without, the fastest idle for 44 % of the launch), neighbouring
    // ids - neighbouring cells of the same frames - are in flight side by side, and the cheap ZERO chunks
    // at the end of the sweep level the tail.  work[1] counts CTAs that are done; the last one rewinds both.
    // The last resampled tiles of the sweep, [split_first, split_end), are handed out in `split` chunks of a
    // fraction of the block's frames each: whoever ends up with the last big chunks holds the launch up by
    // less, and the cheap COPY / ZERO chunks behind them fill the rest of the gap.
    unsigned* work;
    int claim;
    int n_tiles;
    int n_chunks;                       // n_blocks * chunks_per_block
    int chunks_per_block;               // n_tiles + (split_end - split_first) * (split - 1)
    int split_first, split_end, split;
    int light_every, light_end, heavy_end, n_heavy;   // the sweep order inside a block, see decode_chunk
    int frame_block;
    int nf_last;
    int n_blocks;
    int class_first[MCS_N_CLASSES + 1];
    // group descriptors of the FAST tiles (tiles [0, class_first[1])), see mcs_common.h
    int layer_sp[MCS_MAX_LAYERS];       // staged box pitch of each layer in bytes (McsLayer::bw4 * 4)
    int layer_ox[MCS_MAX_LAYERS];       // McsLayer::ox
    const uint8_t* fast;
    int fast_stride;
    int fast_passes;
    int use_fast;                       // 0: this launch's output alignment rules the group path out; FAST
                                        // tiles are then resampled through their per-pixel descriptors
    // feather mode, fused form: BAND tiles (tiles [0, class_first[1])) blend with up to MCS_BAND_MAX_OVERLAYS outer
    // layers, one more staged box per layer and frame; see mcs_tiles.cu for the records
    const int4* band_issue;             // [n_band][1 + MCS_BAND_MAX_OVERLAYS] {layer, bx, by, box bytes}
    const uint32_t* band_desc;          // [n_band][MCS_BAND_MAX_OVERLAYS][2048] overlay descriptors
    int feather_log2;
    int ov_bytes;                       // shared-memory bytes of the overlay-descriptor buffer (0: no BAND tiles)
};

// ---- PTX wrappers ----------------------------------------------------------------------------
extern __shared__ __align__(128) uint8_t smem[];

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
#ifdef TILED_DEBUG_HANG   // debugging aid: a wait that does not end reports where and traps
#define TILED_HANG_CHECK(n_, what_)                                                                              \
    if (++(n_) > (1u << 26)) {                                                                                   \
        printf("tiled kernel stuck: %s line %d cta %d thread %d\n", what_, __LINE__, blockIdx.x, threadIdx.x);  \
        __trap();                                                                                                \
    }
#else
#define TILED_HANG_CHECK(n_, what_)
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int line = 0) {
    uint32_t done;
#ifdef TILED_DEBUG_HANG
    unsigned spins = 0;
#endif
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
#ifdef TILED_DEBUG_HANG
        if (!done && ++spins > (1u << 22)) {
            printf("tiled kernel stuck: mbarrier wait from line %d cta %d thread %d bar %u parity %u\n", line, blockIdx.x,
                   threadIdx.x, bar, parity);
            __trap();
        }
#endif
    } while (!done);
}
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {   // mbar_wait without the wait
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done != 0;
}
// The box origin must sit on a 16-byte boundary of the source row (c0 * 4 bytes % 16 == 0): the
// TMA unit raises an illegal-instruction fault otherwise.  mcs_tiles.cu places the boxes so.
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const CUtensorMap* map, int c0, int c1, int c2,
                                            uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
        "[%0], [%1, {%2, %3, %4}], [%5];" ::"r"(smem_dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
        : "memory");
}
// Plain (1-D) bulk copy global -> shared, completion counted on an mbarrier like the tensor loads.
// Addresses and size are multiples of 16 bytes.
__device__ __forceinline__ void bulk_g2s(uint32_t smem_dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// Shared-memory accesses by absolute shared-window address held in a register.  `volatile` keeps
// them ordered with barriers and with each other; arithmetic is still scheduled across them.
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
// Same load, but NOT volatile: the compiler may schedule it freely between the instruction that
// produced `addr` and the first use of the result - in particular across the (volatile) staging
// stores of the neighbouring pixels, so that the tap loads of all pixels of a thread are in
// flight together.  Only for the staged source boxes, whose address is laundered through
// order_after_wait() after the mbarrier wait that makes the box visible.
__device__ __forceinline__ uint32_t lds32_box(uint32_t addr) {
    uint32_t v;
    asm("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t order_after_wait(uint32_t addr) {
    asm volatile("" : "+r"(addr)::"memory");
    return addr;
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds16(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts8(uint32_t addr, uint32_t v) {   // stores the low byte of v
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void sts16(uint32_t addr, uint32_t v) {  // stores the low two bytes of v
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t dp2a_lo(uint32_t w, uint32_t p, uint32_t acc) {   // acc + w.h0*p.b0 + w.h1*p.b1
    uint32_t r;
    asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(p), "r"(acc));
    return r;
}
__device__ __forceinline__ uint32_t dp2a_hi(uint32_t w, uint32_t p, uint32_t acc) {   // acc + w.h0*p.b2 + w.h1*p.b3
    uint32_t r;
    asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(w), "r"(p), "r"(acc));
    return r;
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {   // selector nibbles all < 8
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

#define MCS_STG128(p, v) __stcs((p), (v))   // streaming: written once, never re-read

// ---- work split --------------------------------------------------------------------------------
// The scheduler is the producer thread: it claims chunk ids from the global counter, decodes them (once: the
// decode costs a few integer divisions) and publishes them to the CTA through a small ring in shared memory, by
// CTA-local sequence number k = 0, 1, 2 ...  Consumers look at chunk k once `published > k`; a tile of -1 ends
// the CTA.  The producer claims at most two chunks past the one it issues boxes for, and it issues boxes for
// chunk k only after every warp has taken chunk k - 2's record out of its buffer, so a ring of TILED_QD entries
// is never overrun.
#define TILED_QD 32
struct SchedMem {
    int published;       // sequence numbers [0, published) have their id in ids[]
    int pad[3];
    int4 chunk[TILED_QD];   // {tile, frame block, first frame, end frame} of sequence number k at [k % QD]; tile -1 = no more work
};

__device__ __forceinline__ int ld_volatile_shared(uint32_t addr) {
    int v;
    asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}

// Claim state, in registers of the producer thread.
struct Sched {
    int claimed;          // sequence numbers published so far
    int ended;            // the end marker has been published
    int has_pend;         // a claim is in flight: its result is `pend`
    unsigned pend;
};

// Chunk id -> frame block, tile and frames [f0, f1) of the block.  Inside a block the sweep INTERLEAVES the
// resampled tiles (FAST, WARP: bound by the SM) evenly with the COPY and ZERO tiles (bound by DRAM): with the
// classes one after the other every CTA is in the same regime at the same time and the launch costs the sum of
// a compute-bound and a memory-bound phase; interleaved, the copies fill the DRAM time the resampling leaves idle.
__device__ __forceinline__ void decode_chunk(const TiledArgs& a, int id, int& blk, int& t, int& f0, int& f1) {
    blk = a.n_blocks > 1 ? id / a.chunks_per_block : 0;
    const int p = id - blk * a.chunks_per_block;
    const int nf = blk == a.n_blocks - 1 ? a.nf_last : a.frame_block;
    f0 = 0;
    f1 = nf;
    // sweep of a block: [0, light_end) every light_every-th position is a COPY / ZERO tile, the others resampled
    // chunks; [light_end, heavy_end) the resampled chunks that are left; [heavy_end, ...) the light tiles left
    int j;
    if (p < a.light_end) {
        const int g = p / a.light_every;
        if (p - g * a.light_every == a.light_every - 1) {
            t = a.split_end + g;
            return;
        }
        j = p - g;
    } else if (p < a.heavy_end) {
        j = p - a.light_end / a.light_every;
    } else {
        t = a.split_end + (p - a.n_heavy);
        return;
    }
    if (j < a.split_first) {
        t = j;
    } else {
        const int q = (j - a.split_first) / a.split, part = (j - a.split_first) - q * a.split;
        t = a.split_first + q;
        f0 = nf * part / a.split;
        f1 = nf * (part + 1) / a.split;
    }
}

__device__ __forceinline__ int tile_class(const TiledArgs& a, int t) {
    return t < a.class_first[1] ? MCS_TILE_BAND : t < a.class_first[2] ? MCS_TILE_FAST : t < a.class_first[3] ? MCS_TILE_WARP
           : t < a.class_first[4] ? MCS_TILE_COPY : MCS_TILE_ZERO;
}

// Make sure sequence numbers below `upto` are published (or the end marker is).  Producer thread.  One claim
// is kept in flight: the atomic is issued when the previous claim is published and its result read at the
// next call, a chunk later, so the round trip to the counter is not on the thread's critical path.
__device__ __forceinline__ void sched_ensure(const TiledArgs& a, SchedMem* sm, Sched& c, int upto) {
    while (!c.ended && c.claimed < upto) {
        unsigned g0;
        if (c.has_pend) {
            g0 = c.pend;
            c.has_pend = 0;
        } else {
            g0 = atomicAdd(a.work, (unsigned)a.claim);
        }
        for (int i = 0; i < a.claim && !c.ended; ++i) {
            const bool more = g0 + (unsigned)i < (unsigned)a.n_chunks;
            int4 e = make_int4(-1, 0, 0, 0);
            if (more) decode_chunk(a, (int)(g0 + (unsigned)i), e.y, e.x, e.z, e.w);
            sm->chunk[c.claimed % TILED_QD] = e;
            ++c.claimed;
            c.ended = more ? 0 : 1;
        }
        __threadfence_block();
        *reinterpret_cast<volatile int*>(&sm->published) = c.claimed;
    }
    if (!c.ended && !c.has_pend) {
        c.pend = atomicAdd(a.work, (unsigned)a.claim);
        c.has_pend = 1;
    }
}

// ---- resampling ----------------------------------------------------------------------------------
// Frame-invariant sampling state of one output pixel.
struct PxDesc {
    uint32_t off;   // byte offset, inside the staged box, of the aligned word holding tap (sx, sy)
    uint32_t sh;    // funnel-shift amount: its low 5 bits are 8 * byte phase of the tap inside that word
    uint32_t w0;    // tap weights of the upper source row, 64 * (32 - ay) * {32 - ax, ax} as two 16-bit lanes
    uint32_t w1;    // tap weights of the lower source row, 64 * ay * {32 - ax, ax}
};

// Byte-permute selectors that gather the taps of this thread's channels from the 8-byte tap
// window (lo, hi) of one source row:  pair -> [c0 tap0, c0 tap1, c1 tap0, c1 tap1] (one IDP.2A.LO
// and one IDP.2A.HI then serve two channels), rest -> the remaining channel(s).
struct TapSel {
    uint32_t pair, rest;
};

// Selectors for staging parity `par` (C == 3: the channels are produced in the order
// (par, par + 1, par + 2) mod 3, see stage_px; otherwise in natural order).
template <int C>
__device__ __forceinline__ TapSel tap_sel(uint32_t par) {
    TapSel s;
    if (C == 3) {
        const uint32_t c0 = par, c1 = par + 1, c2 = par + 2 >= 3 ? par - 1 : par + 2;
        s.pair = c0 | ((3 + c0) << 4) | (c1 << 8) | ((3 + c1) << 12);
        s.rest = (c2 | ((3 + c2) << 4)) * 0x0101u;
    } else if (C == 4) {
        s.pair = 0x5140u;
        s.rest = 0x7362u;
    } else {
        s.pair = 0x3210u;
        s.rest = 0x3210u;
    }
    return s;
}

// One pixel of one frame: value k in bits 16..23 of t[k] (other bits are garbage), where value k is
// the k-th channel in the order of `sel`.
//   value = (sum_taps wy*wx*p * 32 + 16384) >> 15 = (sum_taps (64*wy*wx) * p + 32768) >> 16
// The four 16-bit tap weights 64*wy*wx are frame-invariant (PxDesc), so a channel costs two
// IDP.2A per pixel and frame, chained through the accumulator.
// SP = box pitch in bytes when known at compile time (the second source row then costs no
// address arithmetic), 0 = use `sp`.
template <int C, int SP>
__device__ __forceinline__ void sample_px(uint32_t box, uint32_t sp, const PxDesc& d, const TapSel& sel,
                                          uint32_t (&t)[C]) {
    const uint32_t a0 = box + d.off;
    const uint32_t a1 = SP != 0 ? a0 + SP : a0 + sp;
    if (C == 4) {
        const uint32_t lo0 = lds32_box(a0), hi0 = lds32_box(a0 + 4), lo1 = lds32_box(a1), hi1 = lds32_box(a1 + 4);
        const uint32_t p0 = prmt(lo0, hi0, sel.pair), p1 = prmt(lo1, hi1, sel.pair);
        const uint32_t q0 = prmt(lo0, hi0, sel.rest), q1 = prmt(lo1, hi1, sel.rest);
        t[0] = dp2a_lo(d.w1, p1, dp2a_lo(d.w0, p0, 32768u));
        t[1 % C] = dp2a_hi(d.w1, p1, dp2a_hi(d.w0, p0, 32768u));
        t[2 % C] = dp2a_lo(d.w1, q1, dp2a_lo(d.w0, q0, 32768u));
        t[3 % C] = dp2a_hi(d.w1, q1, dp2a_hi(d.w0, q0, 32768u));
    } else if (C == 3) {
        const uint32_t u0 = lds32_box(a0), u1 = lds32_box(a0 + 4), u2 = lds32_box(a0 + 8);
        const uint32_t v0 = lds32_box(a1), v1 = lds32_box(a1 + 4), v2 = lds32_box(a1 + 8);
        const uint32_t lo0 = __funnelshift_r(u0, u1, d.sh), hi0 = __funnelshift_r(u1, u2, d.sh);
        const uint32_t lo1 = __funnelshift_r(v0, v1, d.sh), hi1 = __funnelshift_r(v1, v2, d.sh);
        const uint32_t p0 = prmt(lo0, hi0, sel.pair), p1 = prmt(lo1, hi1, sel.pair);
        const uint32_t q0 = prmt(lo0, hi0, sel.rest), q1 = prmt(lo1, hi1, sel.rest);
        t[0] = dp2a_lo(d.w1, p1, dp2a_lo(d.w0, p0, 32768u));
        t[1 % C] = dp2a_hi(d.w1, p1, dp2a_hi(d.w0, p0, 32768u));
        t[2 % C] = dp2a_lo(d.w1, q1, dp2a_lo(d.w0, q0, 32768u));
    } else {
        const uint32_t u0 = lds32_box(a0), u1 = lds32_box(a0 + 4), v0 = lds32_box(a1), v1 = lds32_box(a1 + 4);
        const uint32_t lo0 = __funnelshift_r(u0, u1, d.sh), lo1 = __funnelshift_r(v0, v1, d.sh);
        t[0] = dp2a_lo(d.w1, lo1, dp2a_lo(d.w0, lo0, 32768u));
    }
}

// Expand a plan-time descriptor word (mcs_tiles.cu: window byte offset | ax << 16 | ay << 21).
__device__ __forceinline__ PxDesc expand_desc(uint32_t w) {
    PxDesc d;
    const uint32_t b = w & 0xffffu, ax = (w >> 16) & 31u, ay = (w >> 21) & 31u;
    const uint32_t iax64 = (32u - ax) << 6, ax64 = ax << 6, iay = 32u - ay;
    d.off = b & ~3u;
    d.sh = b << 3;
    // 64 * 32 * 32 does not fit 16 bits; 65535 gives the same pixel: the tap then carries all the
    // weight and (65535 p + 32768) >> 16 == p for p < 32768
    d.w0 = min(65535u, iay * iax64) | ((iay * ax64) << 16);
    d.w1 = (ay * iax64) | ((ay * ax64) << 16);
    return d;
}

// ---- write-out ---------------------------------------------------------------------------------
// A lane's share of streaming one row segment of a cell (at most 128 * C <= 512 bytes) from
// shared memory to the panorama: lane l moves the l-th 16-byte chunk of the segment, chunks being
// aligned to the DESTINATION, and one byte of the ragged ends (lanes 0..15 the head, 16..31 the
// tail).  All of it depends only on the 16-byte phase of the destination row, so it is computed
// once per chunk when the frame stride keeps that phase.  Destination positions are 32-bit byte
// offsets from the start of the output frame (the launcher checks that a frame is smaller than
// 4 GiB): the frame base is warp-uniform.
struct RowOut {
    uint32_t s_chunk;  // shared address of this lane's 16-byte chunk (WARP cells: absolute and 16-byte
                       // aligned; COPY cells: relative to the staged box, the aligned word below it)
    uint32_t sh;       // COPY cells: 8 * byte phase of the chunk inside that word
    uint32_t s_byte;   // shared address of this lane's ragged-end byte (COPY: relative to the box)
    uint32_t g_chunk;  // frame offsets of both
    uint32_t g_byte;
    bool do_chunk, do_byte;
};

// s_first / g_first: shared address and frame offset of the first byte of the segment, g_phase:
// its global address modulo 16.
__device__ __forceinline__ RowOut row_split(uint32_t s_first, uint32_t g_first, uint32_t g_phase, bool has,
                                            int nbytes, int lane) {
    RowOut r;
    const int al = (int)((16u - g_phase) & 15u);   // bytes to the first 16-byte boundary of the destination
    const int head = min(nbytes, al);
    const int n = has ? (nbytes - head) >> 4 : 0;
    r.do_chunk = lane < n;
    r.s_chunk = s_first + al + (lane << 4);
    r.sh = 0;
    r.g_chunk = g_first + al + (lane << 4);
    const int e = lane < 16 ? lane : head + (n << 4) + lane - 16;
    r.do_byte = has && (lane < 16 ? lane < head : e < nbytes);
    r.s_byte = s_first + e;
    r.g_byte = g_first + e;
    return r;
}

// WARP cells: the staging row has the destination's 16-byte phase, chunks are LDS.128 -> STG.128.
// s_chunk is 16-byte aligned and inside the CTA's shared memory for every lane, so the loads
// need no predicate.  `ragged` (warp-uniform): some lane has a ragged-end byte to move; never
// the case for whole cells of a panorama with 32-byte aligned rows.
__device__ __forceinline__ void write_out(const RowOut& r0, const RowOut& r1, bool ragged, uint8_t* frame) {
    const uint4 v0 = lds128(r0.s_chunk);
    const uint4 v1 = lds128(r1.s_chunk);
    if (r0.do_chunk) MCS_STG128(reinterpret_cast<uint4*>(frame + r0.g_chunk), v0);
    if (r1.do_chunk) MCS_STG128(reinterpret_cast<uint4*>(frame + r1.g_chunk), v1);
    if (ragged) {
        if (r0.do_byte) frame[r0.g_byte] = (uint8_t)lds8(r0.s_byte);
        if (r1.do_byte) frame[r1.g_byte] = (uint8_t)lds8(r1.s_byte);
    }
}

// COPY cells: the staged box keeps the SOURCE's phase, the chunk is realigned with funnel shifts
// (five aligned words cover any 16 bytes; the box is one word wider than the copied window).
__device__ __forceinline__ void copy_out(const RowOut& r, uint32_t box, bool ragged, uint8_t* frame) {
    if (r.do_chunk) {
        const uint32_t w = box + r.s_chunk;
        const uint32_t w0 = lds32(w), w1 = lds32(w + 4), w2 = lds32(w + 8), w3 = lds32(w + 12), w4 = lds32(w + 16);
        uint4 v;
        v.x = __funnelshift_r(w0, w1, r.sh);
        v.y = __funnelshift_r(w1, w2, r.sh);
        v.z = __funnelshift_r(w2, w3, r.sh);
        v.w = __funnelshift_r(w3, w4, r.sh);
        MCS_STG128(reinterpret_cast<uint4*>(frame + r.g_chunk), v);
    }
    if (ragged && r.do_byte) frame[r.g_byte] = (uint8_t)lds8(box + r.s_byte);
}

// Stage the C values of one pixel (bits 16..23 of t[k]) at staging address o.  For C == 3 the
// values were produced in the order (c, c+1, c+2) mod 3 with c = o & 1, so that an aligned
// 16-bit store and one byte store cover the pixel: even o -> [B G] at o, R at o + 2; odd o ->
// B at o, [G R] at o + 1.
template <int C>
__device__ __forceinline__ void stage_px(uint32_t o16, uint32_t o8, const uint32_t (&t)[C]) {
    if (C == 3) {
        sts16(o16, __byte_perm(t[0], t[1], 0x0062));
        sts8(o8, t[2] >> 16);
    } else {
#pragma unroll
        for (int k = 0; k < C; ++k) sts8(o16 + k, t[k] >> 16);
    }
}

// Position in the staging ring.
#define TILED_SCHED_BYTES 640
static_assert(sizeof(SchedMem) <= TILED_SCHED_BYTES, "SchedMem must fit its shared-memory slot");

// Chunk records: while a chunk is being processed the tile record and the descriptors of the NEXT
// one are copied into one of two shared-memory buffers by the bulk-copy engine, so that a chunk
// starts without a global-memory round trip (two dependent ones, tile then descriptors, used to
// cost ~0.9 us of CTA time per chunk and forced long chunks, i.e. large frame blocks).
// Buffer layout: [McsTile, 32 B][FAST: list lengths, 8 B][pad to 64][descriptors].
#define TILED_DESC_BUF_BYTES (MCS_FAST_HEADER_BYTES + MCS_CELL_W * MCS_CELL_H * 4)
static_assert(MCS_FAST_GROUP_BYTES + MCS_FAST_MAX_PASSES * MCS_FAST_PASS_BYTES <= MCS_CELL_W * MCS_CELL_H * 4,
              "a FAST record must fit the chunk-record buffer");

struct RingPos {
    int slot;
    uint32_t phase;
    int n;   // boxes consumed so far
    __device__ __forceinline__ void advance(int stages) {
        ++n;
        if (++slot == stages) { slot = 0; phase ^= 1; }
    }
};

// Shared-memory geometry of a CTA, all as shared-window addresses.
struct Smem {
    uint32_t base;      // ring of `stages` boxes
    uint32_t out;       // staging 16 x OUT_PITCH
    uint32_t full;      // full barriers
    uint32_t empty;     // empty barriers
    uint32_t dbar;      // chunk-record barriers: full[2] at +0, +8, empty[2] at +16, +24; at +32, +48 the
                        // {frame block, first frame, end frame} of the chunk in each buffer
    uint32_t dbuf;      // two chunk-record buffers of TILED_DESC_BUF_BYTES
    uint32_t ov;        // BAND tiles: overlay descriptors of the chunk being processed (MCS_BAND_MAX_OVERLAYS slabs),
                        // behind them its full barrier (+0) and its empty barrier (+8)
    SchedMem* sched;    // chunk ids claimed by the producer
};

// Start the copy of the record of chunk e = {tile, frame block, first frame, end frame} into buffer b, and
// leave the chunk's frames there for the consumers (the store is ordered before their wait by the barrier
// arrive).  One thread.
__device__ __forceinline__ void prefetch_chunk(const TiledArgs& a, const Smem& sm, int b, int4 e) {
    const int t = e.x;
    sts32(sm.dbar + 32 + 16 * b, (uint32_t)e.y);
    sts32(sm.dbar + 36 + 16 * b, (uint32_t)e.z);
    sts32(sm.dbar + 40 + 16 * b, (uint32_t)e.w);
    const int cls = tile_class(a, t);
    const uint32_t dst = sm.dbuf + b * TILED_DESC_BUF_BYTES, bar = sm.dbar + 8 * b;
    if (cls == MCS_TILE_FAST && a.use_fast) {
        mbar_expect_tx(bar, (uint32_t)a.fast_stride);
        bulk_g2s(dst, a.fast + (size_t)(t - a.class_first[1]) * a.fast_stride, (uint32_t)a.fast_stride, bar);
    } else if (cls >= MCS_TILE_WARP) {
        mbar_expect_tx(bar, 32u + MCS_CELL_W * MCS_CELL_H * 4u);
        bulk_g2s(dst, a.tiles + t, 32u, bar);
        bulk_g2s(dst + MCS_FAST_HEADER_BYTES, a.desc + (size_t)t * (MCS_CELL_W * MCS_CELL_H), MCS_CELL_W * MCS_CELL_H * 4u, bar);
    } else {
        mbar_expect_tx(bar, 32u);
        bulk_g2s(dst, a.tiles + t, 32u, bar);
    }
}

// The producer: one thread, lane 0 of the first warp behind the resampling warps.  Per chunk in claim order
// it issues the chunk's boxes, one per frame (BAND tiles: one per layer involved and frame, the owner's first
// unless the tile is zero-base), each as soon as its slot is released; in between it starts the copy of the
// NEXT chunk's record once every warp is done with the buffer, and waits for that buffer only when all boxes
// of the chunk are out.  Both waits are deadlock-free: a warp that holds a slot or a record buffer is in a
// chunk whose boxes and record are already on their way.  tests/test_producer_protocol.py restates this.
template <bool BANDS>
__device__ __forceinline__ void produce(const TiledArgs& a, const Smem& sm) {
    SchedMem* const q = sm.sched;
    Sched c{0, 0, 0, 0u};
    sched_ensure(a, q, c, 1);
    if (q->chunk[0].x >= 0) prefetch_chunk(a, sm, 0, q->chunk[0]);
    int slot = 0;
    uint32_t phase = 0;
    for (int k = 0;; ++k) {
        sched_ensure(a, q, c, k + 2);
        const int4 e = q->chunk[k % TILED_QD];
        if (e.x < 0) break;
        // the record of chunk k + 1 (published: e is not the end marker) still has to be copied; its buffer last
        // held chunk k - 1 (none for k == 0)
        bool rec_todo = q->chunk[(k + 1) % TILED_QD].x >= 0;
        const uint32_t rel = sm.dbar + 16 + 8 * ((k + 1) & 1), rel_par = (uint32_t)(((k - 1) >> 1) & 1);
        if (e.x < a.class_first[MCS_N_CLASSES - 1]) {   // ZERO chunks stage nothing
            // the box records are re-read per box (L1 hits) rather than held in the producer's 32 registers
            const int w = __ldg(&a.issue[e.x].w);
            const int nl = BANDS ? 1 + ((w >> 24) & 15) : 1, li0 = BANDS ? (w >> 28) & 1 : 0;
            const int frame0 = e.y * a.frame_block;
            for (int f = e.z; f < e.w; ++f) {
                for (int li = li0; li < nl; ++li) {
                    int4 r = __ldg(BANDS && li > 0 ? a.band_issue + e.x * (1 + MCS_BAND_MAX_OVERLAYS) + li : a.issue + e.x);
                    if (!(BANDS && li > 0)) r.w &= 0xffffff;
                    if (rec_todo && (k == 0 || mbar_test(rel, rel_par))) {
                        prefetch_chunk(a, sm, (k + 1) & 1, q->chunk[(k + 1) % TILED_QD]);
                        rec_todo = false;
                    }
                    mbar_wait(sm.empty + 8 * slot, phase ^ 1, __LINE__);   // first trip round the ring: passes at once
                    mbar_expect_tx(sm.full + 8 * slot, (uint32_t)r.w);
                    tma_load_3d(sm.base + slot * a.box_bytes, &a.tmap[r.x], r.y, r.z, frame0 + f, sm.full + 8 * slot);
                    if (++slot == a.stages) { slot = 0; phase ^= 1; }
                }
            }
        }
        if (rec_todo) {
            if (k >= 1) mbar_wait(rel, rel_par, __LINE__);
            prefetch_chunk(a, sm, (k + 1) & 1, q->chunk[(k + 1) % TILED_QD]);
        }
    }
    // every CTA ends on a claim past the last chunk; the last CTA out rewinds the counters for the next launch
    __threadfence();
    if (atomicAdd(a.work + 1, 1u) == gridDim.x - 1) {
        a.work[0] = 0u;
        a.work[1] = 0u;
        __threadfence();
    }
}

// The n_fr frames of one WARP chunk for one warp: per frame wait for the staged box, resample
// this thread's (up to) 8 pixels into the warp's two staging rows, release the box, stream the
// rows out.  `groups` has bit j set when pixel group j of this warp (row j>>2, columns
// 32*(j&3) .. +31) contains owned pixels; it is warp-uniform.  frame = first output frame,
// g_row0 = frame offset of column 0 of cell row `warp`.
// BAND: the tile blends with n_ov outer layers (feather mode): after the owner's pixels are staged, each overlay
// box is waited for in turn and the pixels its descriptors mark (sm.ov, slab o; box pitch ov_sp[o]) are resampled
// from it and blended into the staged values - value = (a * value + (F - a) * sample + F/2) >> feather_log2 -
// before the rows go out.
template <int C, int SP, bool BAND>
__device__ __forceinline__ void warp_frames(const TiledArgs& a, const PxDesc (&d)[8], uint32_t groups, uint32_t sp,
                                            const Smem& sm, RingPos& ring, uint8_t* frame,
                                            uint32_t g_row0, int n_fr, int c0, int nbytes, int h, int warp,
                                            int lane, int n_ov = 0, uint32_t ov_sp0 = 0, uint32_t ov_sp1 = 0,
                                            bool zero_base = false) {
    // BAND: which of this warp's eight pixel slots hold blended pixels, per overlay (bits 8 o .. 8 o + 7; warp-uniform)
    uint32_t ov_slots = 0;
    if (BAND) {
        for (int o = 0; o < n_ov; ++o)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t w = lds32(sm.ov + (uint32_t)o * (MCS_CELL_W * MCS_CELL_H * 4) + ((j * TILED_WARPS + warp) * 32 + lane) * 4);
                if (__any_sync(0xffffffffu, (w >> 26) != 0u)) ov_slots |= 1u << (8 * o + j);
            }
    }
    constexpr int OUT_PITCH = MCS_CELL_W * C + 16;
    const int stages = a.stages;
    const uint32_t g_row1 = g_row0 + (uint32_t)TILED_WARPS * (uint32_t)a.dst_pitch;
    const uint32_t s_row0 = sm.out + warp * OUT_PITCH, s_row1 = s_row0 + TILED_WARPS * OUT_PITCH;
    const bool has0 = warp < h, has1 = warp + TILED_WARPS < h;
    const bool phase_moves = (a.dst_frame_stride & 15) != 0;   // the rows' 16-byte phase differs per frame

    // Staging rows carry the 16-byte phase of the destination row (column 0), so that the
    // segment [c0, c1) is copied out with aligned 16-byte loads and stores.
    uint32_t ph0 = ((uint32_t)reinterpret_cast<uintptr_t>(frame) + g_row0) & 15u;
    uint32_t ph1 = ((uint32_t)reinterpret_cast<uintptr_t>(frame) + g_row1) & 15u;
    RowOut r0 = row_split(s_row0 + ph0 + c0 * C, g_row0 + c0 * C, (ph0 + c0 * C) & 15u, has0, nbytes, lane);
    RowOut r1 = row_split(s_row1 + ph1 + c0 * C, g_row1 + c0 * C, (ph1 + c0 * C) & 15u, has1, nbytes, lane);
    // staging addresses and channel order of this thread's pixels (rows 8 apart share the parity
    // of their phase, so one channel order serves both)
    uint32_t st0 = s_row0 + ph0 + lane * C, st1 = s_row1 + ph1 + lane * C;
    uint32_t par = C == 3 ? (st0 & 1u) : 0u;
    TapSel sel = tap_sel<C>(par);
    bool ragged = __any_sync(0xffffffffu, r0.do_byte || r1.do_byte);

    for (int i = 0; i < n_fr; ++i, frame += a.dst_frame_stride) {
        if (phase_moves && i != 0) {
            ph0 = ((uint32_t)reinterpret_cast<uintptr_t>(frame) + g_row0) & 15u;
            ph1 = ((uint32_t)reinterpret_cast<uintptr_t>(frame) + g_row1) & 15u;
            r0 = row_split(s_row0 + ph0 + c0 * C, g_row0 + c0 * C, (ph0 + c0 * C) & 15u, has0, nbytes, lane);
            r1 = row_split(s_row1 + ph1 + c0 * C, g_row1 + c0 * C, (ph1 + c0 * C) & 15u, has1, nbytes, lane);
            st0 = s_row0 + ph0 + lane * C;
            st1 = s_row1 + ph1 + lane * C;
            ragged = __any_sync(0xffffffffu, r0.do_byte || r1.do_byte);
            if (C == 3) {
                par = st0 & 1u;
                sel = tap_sel<C>(par);
            }
        }
        // even staging address: 16-bit store at +0, byte at +2; odd: byte at +0, 16-bit store at +1
        const uint32_t o16_0 = st0 + par, o8_0 = st0 + 2 - 2 * par;
        const uint32_t o16_1 = st1 + par, o8_1 = st1 + 2 - 2 * par;

        if (BAND && zero_base) {
            // the owner contributes nothing to this tile: no box of it was staged, the overlays blend into zeros
            uint32_t z[C];
#pragma unroll
            for (int k = 0; k < C; ++k) z[k] = 0u;
#pragma unroll
            for (int j8 = 0; j8 < 8; ++j8) {
                const int g = 32 * (j8 & 3) * C;
                stage_px<C>((j8 < 4 ? o16_0 : o16_1) + g, (j8 < 4 ? o8_0 : o8_1) + g, z);
            }
            __syncwarp();
        } else {
        mbar_wait(sm.full + 8 * ring.slot, ring.phase, __LINE__);
        const uint32_t box = order_after_wait(sm.base + ring.slot * a.box_bytes);
        if (groups == 0xffu) {
            // All tap loads and arithmetic of a batch of pixels come before its first staging
            // store: ptxas cannot prove that a store does not alias a later load, so stores in
            // between would serialise the pixels' (long) dependency chains.
#pragma unroll
            for (int b = 0; b < 8; b += TILED_PX_BATCH) {
                uint32_t t[TILED_PX_BATCH][C];
#pragma unroll
                for (int j = 0; j < TILED_PX_BATCH; ++j) sample_px<C, SP>(box, sp, d[b + j], sel, t[j]);
#pragma unroll
                for (int j = 0; j < TILED_PX_BATCH; ++j) {
                    const int g = 32 * ((b + j) & 3) * C;
                    stage_px<C>((b + j < 4 ? o16_0 : o16_1) + g, (b + j < 4 ? o8_0 : o8_1) + g, t[j]);
                }
            }
        } else {
#pragma unroll 1
            for (int jj = 0; jj < 4; ++jj) {   // pairs (row 0, row 1) of one column group
                if (!(groups & (0x11u << jj))) continue;
                uint32_t t0[C], t1[C];
                const PxDesc da = jj == 0 ? d[0] : jj == 1 ? d[1] : jj == 2 ? d[2] : d[3];
                const PxDesc db = jj == 0 ? d[4] : jj == 1 ? d[5] : jj == 2 ? d[6] : d[7];
                sample_px<C, SP>(box, sp, da, sel, t0);
                sample_px<C, SP>(box, sp, db, sel, t1);
                const int g = 32 * jj * C;
                stage_px<C>(o16_0 + g, o8_0 + g, t0);
                stage_px<C>(o16_1 + g, o8_1 + g, t1);
            }
        }
        __syncwarp();   // every lane has consumed its box reads and staged its pixels
        if (lane == 0) mbar_arrive(sm.empty + 8 * ring.slot);
        ring.advance(stages);
        }

        if (BAND) {
            const uint32_t F = 1u << a.feather_log2;
#pragma unroll 1
            for (int o = 0; o < n_ov; ++o) {
                mbar_wait(sm.full + 8 * ring.slot, ring.phase, __LINE__);
                const uint32_t obox = order_after_wait(sm.base + ring.slot * a.box_bytes);
                const uint32_t osp = o == 0 ? ov_sp0 : ov_sp1;
                const uint32_t slab = sm.ov + (uint32_t)o * (MCS_CELL_W * MCS_CELL_H * 4) + (warp * 32 + lane) * 4;
#pragma unroll 1
                for (uint32_t todo = (ov_slots >> (8 * o)) & 0xffu; todo != 0u; todo &= todo - 1u) {
                    const int j = __ffs((int)todo) - 1;
                    const uint32_t w = lds32(slab + j * (TILED_WARPS * 32 * 4));
                    if (w >> 26) {
                        const uint32_t wa = (w >> 26) - 1u, wb = F - wa;   // weights of the staged value / the sample
                        const PxDesc dd = expand_desc(w & 0x03ffffffu);
                        uint32_t t[C];
                        sample_px<C, 0>(obox, osp, dd, sel, t);
                        const int g = 32 * (j & 3) * C;
                        const uint32_t p16 = (j < 4 ? o16_0 : o16_1) + g, p8 = (j < 4 ? o8_0 : o8_1) + g;
                        uint32_t v[C];
                        if (C == 3) {
                            const uint32_t lo = lds16(p16);
                            v[0] = lo & 0xffu;
                            v[1 % C] = lo >> 8;
                            v[2 % C] = lds8(p8);
                        } else {
#pragma unroll
                            for (int k = 0; k < C; ++k) v[k] = lds8(p16 + k);
                        }
#pragma unroll
                        for (int k = 0; k < C; ++k)
                            t[k] = ((wa * v[k] + wb * ((t[k] >> 16) & 0xffu) + (F >> 1)) >> a.feather_log2) << 16;
                        stage_px<C>(p16, p8, t);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(sm.empty + 8 * ring.slot);
                ring.advance(stages);
            }
        }

        write_out(r0, r1, ragged, frame);
        __syncwarp();   // staging rows are rewritten by the next frame
    }
}

// ---- group resampling (FAST tiles, C == 3) -------------------------------------------------------
// Thread (warp, lane) owns, in each of its two cell rows, the four adjacent pixels at cell columns
// 4 lane .. 4 lane + 3.  When they sample four adjacent source pixels of one source row pair - the
// rule at near-unit scale - their taps are the 15 bytes after the group's anchor in each of the
// two source rows: five aligned words per row, realigned to the anchor with four funnel shifts,
// serve all four pixels through byte permutes with CONSTANT selectors (pixel j's taps start 3 j
// bytes after the anchor), and the twelve output bytes leave as three aligned 32-bit stores.
// Against the per-pixel path that is 10 instead of 24 tap loads, 8 instead of 16 funnel shifts
// and 3 instead of 8 staging stores per four pixels.  Pixels that do not fit the template (the
// source column or row slips inside the group) are listed per warp at plan time (mcs_tiles.cu)
// and resampled by one or two extra per-pixel passes, lane l taking entries l and 32 + l.
struct GroupDesc {
    uint32_t off;     // byte offset, inside the staged box, of the aligned word holding the anchor tap
    uint32_t sh;      // 8 * byte phase of the anchor inside that word
    uint32_t w0[4];   // per pixel: tap weights of the upper / lower source row (as PxDesc)
    uint32_t w1[4];
};

__device__ __forceinline__ void tap_weights(uint32_t ax, uint32_t ay, uint32_t& w0, uint32_t& w1) {
    const uint32_t iax64 = (32u - ax) << 6, ax64 = ax << 6, iay = 32u - ay;
    w0 = min(65535u, iay * iax64) | ((iay * ax64) << 16);   // see expand_desc
    w1 = (ay * iax64) | ((ay * ax64) << 16);
}

__device__ __forceinline__ GroupDesc expand_group(uint2 g) {
    GroupDesc d;
    const uint32_t b = g.x & 0xffffu;
    d.off = b & ~3u;
    d.sh = (b & 3u) << 3;
    tap_weights((g.x >> 16) & 31u, (g.x >> 21) & 31u, d.w0[0], d.w1[0]);
#pragma unroll
    for (int j = 1; j < 4; ++j)
        tap_weights((g.y >> (10 * (j - 1))) & 31u, (g.y >> (10 * (j - 1) + 5)) & 31u, d.w0[j], d.w1[j]);
    return d;
}

// byte 2 of a, b, c, d as one word
__device__ __forceinline__ uint32_t pack4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    return prmt(prmt(a, b, 0x6262u), prmt(c, d, 0x6262u), 0x5410u);
}

// The four pixels of a group for one frame: twelve output bytes in memory order.
template <int SP>
__device__ __forceinline__ void sample_group(uint32_t box, uint32_t sp, const GroupDesc& d, uint32_t (&out)[3]) {
    const uint32_t a0 = box + d.off;
    const uint32_t a1 = SP != 0 ? a0 + SP : a0 + sp;
    uint32_t u[5], v[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        u[i] = lds32_box(a0 + 4 * i);
        v[i] = lds32_box(a1 + 4 * i);
    }
    uint32_t A[4], B[4];   // the rows' bytes from the anchor on
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        A[i] = __funnelshift_r(u[i], u[i + 1], d.sh);
        B[i] = __funnelshift_r(v[i], v[i + 1], d.sh);
    }
    uint32_t t[4][3];
    // pixel j: taps at bytes 3 j .. 3 j + 5; selectors relative to the word pair (k, k + 1)
#define MCS_GROUP_PX(j, k, selp, kq, selq)                                                   \
    {                                                                                        \
        const uint32_t p0 = prmt(A[k], A[k + 1], selp), p1 = prmt(B[k], B[k + 1], selp);     \
        const uint32_t q0 = prmt(A[kq], A[kq + 1], selq), q1 = prmt(B[kq], B[kq + 1], selq); \
        t[j][0] = dp2a_lo(d.w1[j], p1, dp2a_lo(d.w0[j], p0, 32768u));                        \
        t[j][1] = dp2a_hi(d.w1[j], p1, dp2a_hi(d.w0[j], p0, 32768u));                        \
        t[j][2] = dp2a_lo(d.w1[j], q1, dp2a_lo(d.w0[j], q0, 32768u));                        \
    }
    MCS_GROUP_PX(0, 0, 0x4130u, 0, 0x5252u)   // bytes 0..5
    MCS_GROUP_PX(1, 0, 0x7463u, 1, 0x4141u)   // bytes 3..8
    MCS_GROUP_PX(2, 1, 0x6352u, 1, 0x7474u)   // bytes 6..11
    MCS_GROUP_PX(3, 2, 0x5241u, 2, 0x6363u)   // bytes 9..14
#undef MCS_GROUP_PX
    out[0] = pack4(t[0][0], t[0][1], t[0][2], t[1][0]);
    out[1] = pack4(t[1][1], t[1][2], t[2][0], t[2][1]);
    out[2] = pack4(t[2][2], t[3][0], t[3][1], t[3][2]);
}

// One entry of a warp's general list for this lane.
struct GenDesc {
    PxDesc d;
    uint32_t pos;   // slot << 31 | valid << 30 | (staging byte offset relative to the lane's own group) & 0xffff
};

__device__ __forceinline__ GenDesc expand_gen(uint2 e, int lane) {
    GenDesc g;
    g.d = expand_desc(e.x);
    const int rel = (int)(e.y & 127u) * 3 - lane * 12;
    g.pos = e.y == 0xffffffffu ? 0u : ((e.y & 128u) << 24) | 0x40000000u | ((uint32_t)rel & 0xffffu);
    return g;
}

// The n_fr frames of one FAST chunk for one warp (the group-path counterpart of warp_frames).  The
// caller passes single frames when the rows' 16-byte phase differs from frame to frame.
template <int SP>
__device__ __forceinline__ void fast_frames(const TiledArgs& a, const GroupDesc& g0, const GroupDesc& g1,
                                            const GenDesc (&gen)[MCS_FAST_MAX_PASSES], int n_pass, uint32_t sp,
                                            const Smem& sm, RingPos& ring, uint8_t* frame,
                                            uint32_t g_row0, int n_fr, int c0, int nbytes, int h, int warp,
                                            int lane) {
    constexpr int C = 3;
    constexpr int OUT_PITCH = MCS_CELL_W * C + 16;
    const int stages = a.stages;
    const TapSel sel = tap_sel<C>(0u);
    RowOut r0, r1;
    uint32_t st0, st1;
    bool ragged;
    {
        const uint32_t g_row1 = g_row0 + (uint32_t)TILED_WARPS * (uint32_t)a.dst_pitch;
        const uint32_t s_row0 = sm.out + warp * OUT_PITCH, s_row1 = s_row0 + TILED_WARPS * OUT_PITCH;
        // the launcher admits the group path only for 4-byte aligned output rows: ph0, ph1 are multiples of 4
        const uint32_t ph0 = ((uint32_t)reinterpret_cast<uintptr_t>(frame) + g_row0) & 15u;
        const uint32_t ph1 = ((uint32_t)reinterpret_cast<uintptr_t>(frame) + g_row1) & 15u;
        r0 = row_split(s_row0 + ph0 + c0 * C, g_row0 + c0 * C, (ph0 + c0 * C) & 15u, warp < h, nbytes, lane);
        r1 = row_split(s_row1 + ph1 + c0 * C, g_row1 + c0 * C, (ph1 + c0 * C) & 15u, warp + TILED_WARPS < h, nbytes,
                       lane);
        st0 = s_row0 + ph0 + lane * (4 * C);
        st1 = s_row1 + ph1 + lane * (4 * C);
        ragged = __any_sync(0xffffffffu, r0.do_byte || r1.do_byte);
    }
    for (int i = 0; i < n_fr; ++i, frame += a.dst_frame_stride) {
        mbar_wait(sm.full + 8 * ring.slot, ring.phase, __LINE__);
        const uint32_t box = order_after_wait(sm.base + ring.slot * a.box_bytes);
        {
            uint32_t o0[3], o1[3];
            sample_group<SP>(box, sp, g0, o0);
            sample_group<SP>(box, sp, g1, o1);
            sts32(st0, o0[0]); sts32(st0 + 4, o0[1]); sts32(st0 + 8, o0[2]);
            sts32(st1, o1[0]); sts32(st1 + 4, o1[1]); sts32(st1 + 8, o1[2]);
        }
        if (n_pass > 0) {
            __syncwarp();   // a general pixel replaces bytes another lane's group store just wrote
#pragma unroll
            for (int p = 0; p < MCS_FAST_MAX_PASSES; ++p) {
                if (p < n_pass) {
                    uint32_t t[C];
                    sample_px<C, SP>(box, sp, gen[p].d, sel, t);
                    const uint32_t o = ((int)gen[p].pos < 0 ? st1 : st0) + (uint32_t)(int)(short)gen[p].pos;
                    if (gen[p].pos & 0x40000000u) {
                        sts8(o, t[0] >> 16);
                        sts8(o + 1, t[1] >> 16);
                        sts8(o + 2, t[2] >> 16);
                    }
                }
            }
        }
        __syncwarp();   // every lane has consumed its box reads and staged its pixels
        if (lane == 0) mbar_arrive(sm.empty + 8 * ring.slot);
        ring.advance(stages);

        write_out(r0, r1, ragged, frame);
        __syncwarp();   // staging rows are rewritten by the next frame
    }
}

template <int C, bool BANDS>
__global__ void __launch_bounds__(TILED_CTA_THREADS, TILED_MIN_CTAS)
mcs_stitch_tiled_kernel(const __grid_constant__ TiledArgs a) {
    constexpr int OUT_PITCH = MCS_CELL_W * C + 16;
    // layout: [ring of `stages` boxes][full barriers][empty barriers][chunk ids][chunk-record barriers]
    //         [staging 16 x OUT_PITCH][two chunk-record buffers][slack]
    // (slack: the unpredicated 16-byte loads of write_out start up to 15 + 127 C + 15 + 496 bytes
    // past the start of a staging row, i.e. up to ~1 KB past the start of the last row)
    const int stages = a.stages;
    Smem sm;
    sm.base = smem_u32(smem);
    sm.full = sm.base + stages * a.box_bytes;
    sm.empty = sm.full + 8 * TILED_MAX_STAGES;
    sm.sched = reinterpret_cast<SchedMem*>(smem + stages * a.box_bytes + 16 * TILED_MAX_STAGES);
    sm.dbar = sm.empty + 8 * TILED_MAX_STAGES + TILED_SCHED_BYTES;
    sm.out = sm.dbar + 64;
    sm.dbuf = (sm.out + MCS_CELL_H * OUT_PITCH + 15u) & ~15u;
    sm.ov = sm.dbuf + 2 * TILED_DESC_BUF_BYTES + 1024;   // behind the slack of the write-out loads
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        sm.sched->published = 0;
        for (int s = 0; s < stages; ++s) {
            mbar_init(sm.full + 8 * s, 1);
            mbar_init(sm.empty + 8 * s, TILED_WARPS);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(sm.dbar + 8 * b, 1);
            mbar_init(sm.dbar + 16 + 8 * b, TILED_WARPS);
        }
        if (BANDS) {
            mbar_init(sm.ov + a.ov_bytes, 1);
            mbar_init(sm.ov + a.ov_bytes + 8, TILED_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    if (warp >= TILED_WARPS) {   // the producer warpgroup
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(TILED_PRODUCER_REGS));
        if (tid == TILED_THREADS) produce<BANDS>(a, sm);
        return;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(TILED_CONSUMER_REGS));
    // keep the shared-window addresses in registers: left alone, the compiler rematerialises them
    // in the frame loop from SR_CgaCtaId and the kernel parameters
    asm volatile("" : "+r"(sm.base), "+r"(sm.full), "+r"(sm.empty), "+r"(sm.out));

    RingPos ring{0, 0u, 0};
    if (BANDS && lane == 0) sts32(sm.ov + a.ov_bytes + 16 + 4 * warp, 0u);   // BAND chunks this warp has processed (phase of the overlay buffer's barriers; own warp only)
    const uint32_t s_published = smem_u32(&sm.sched->published), s_ids = smem_u32(&sm.sched->chunk[0]);
    for (int k_cons = 0;; ++k_cons) {
        // ---- chunk record: wait for this chunk's ----
        const int cb = k_cons & 1;
        const uint32_t rec = sm.dbuf + cb * TILED_DESC_BUF_BYTES;
        const uint32_t rec_release = sm.dbar + 16 + 8 * cb;
        {
#ifdef TILED_DEBUG_HANG
            unsigned spins = 0;
#endif
            while (ld_volatile_shared(s_published) <= k_cons) { TILED_HANG_CHECK(spins, "waiting for a chunk id") }
        }
        const int id = ld_volatile_shared(s_ids + 16 * (k_cons % TILED_QD));   // the chunk's tile
        if (id < 0) break;
        mbar_wait(sm.dbar + 8 * cb, (uint32_t)((k_cons >> 1) & 1), __LINE__);
        const uint4 info = lds128(sm.dbar + 32 + 16 * cb);
        const int blk = (int)info.x, f0 = (int)info.y, f1 = (int)info.z;
        McsTile tile;
        {
            const uint4 q0 = lds128(rec), q1 = lds128(rec + 16);
            tile.cx0 = (int)q0.x;
            tile.y0 = (int)q0.y;
            tile.c0 = (short)(q0.z & 0xffffu);
            tile.c1 = (short)(q0.z >> 16);
            tile.h = (short)(q0.w & 0xffffu);
            tile.layer = (short)(q0.w >> 16);
            tile.cls = (short)(q1.x & 0xffffu);
            tile.flags = (short)(q1.x >> 16);
            tile.bx = (int)q1.y;
            tile.by = (int)q1.z;
            tile.reserved = (int)q1.w;
        }
        const int c0 = tile.c0, c1 = tile.c1, h = tile.h;
        const int nbytes = (c1 - c0) * C;
        const int n_fr = f1 - f0;
        // first output frame of the chunk (warp-uniform)
        uint8_t* const frame0 = a.dst + ((long long)blk * a.frame_block + f0) * a.dst_frame_stride;
        // frame offset of cell column 0, row 0 (modulo 2^32: the column may lie left of the row, the
        // owned columns never do)
        const uint32_t g_cell = (uint32_t)tile.y0 * (uint32_t)a.dst_pitch + (uint32_t)(tile.cx0 * C);
        const bool phase_moves = (a.dst_frame_stride & 15) != 0;

        if (tile.cls == MCS_TILE_ZERO || tile.cls == MCS_TILE_COPY) {   // nothing more to read from the chunk record
            __syncwarp();
            if (lane == 0) mbar_arrive(rec_release);
        }
        if (tile.cls == MCS_TILE_ZERO) {
            const uint32_t g_first0 = g_cell + (uint32_t)warp * (uint32_t)a.dst_pitch + c0 * C;
            const uint32_t g_first1 = g_first0 + (uint32_t)TILED_WARPS * (uint32_t)a.dst_pitch;
            uint8_t* frame = frame0;
            RowOut r0, r1;
            for (int i = 0; i < n_fr; ++i, frame += a.dst_frame_stride) {
                if (i == 0 || phase_moves) {
                    const uint32_t fp = (uint32_t)reinterpret_cast<uintptr_t>(frame);
                    r0 = row_split(0, g_first0, (fp + g_first0) & 15u, warp < h, nbytes, lane);
                    r1 = row_split(0, g_first1, (fp + g_first1) & 15u, warp + TILED_WARPS < h, nbytes, lane);
                }
                const uint4 z = make_uint4(0u, 0u, 0u, 0u);
                if (r0.do_chunk) MCS_STG128(reinterpret_cast<uint4*>(frame + r0.g_chunk), z);
                if (r1.do_chunk) MCS_STG128(reinterpret_cast<uint4*>(frame + r1.g_chunk), z);
                if (r0.do_byte) frame[r0.g_byte] = 0;
                if (r1.do_byte) frame[r1.g_byte] = 0;
            }
            continue;
        }
        const uint32_t sp = (uint32_t)a.layer_sp[tile.layer];

        if (tile.cls == MCS_TILE_COPY) {
            // rows warp and warp + 8 of the cell; everything but the box address is frame-invariant
            const uint32_t s_off = (uint32_t)((tile.cx0 + c0 - a.layer_ox[tile.layer]) * C - 4 * tile.bx);   // first byte inside the box row
            const uint32_t g_first0 = g_cell + (uint32_t)warp * (uint32_t)a.dst_pitch + c0 * C;
            const uint32_t g_first1 = g_first0 + (uint32_t)TILED_WARPS * (uint32_t)a.dst_pitch;
            uint8_t* frame = frame0;
            RowOut r0, r1;
            bool ragged = false;
            for (int i = 0; i < n_fr; ++i, frame += a.dst_frame_stride) {
                if (i == 0 || phase_moves) {
                    const uint32_t fp = (uint32_t)reinterpret_cast<uintptr_t>(frame);
                    r0 = row_split(s_off + warp * sp, g_first0, (fp + g_first0) & 15u, warp < h, nbytes, lane);
                    r1 = row_split(s_off + (warp + TILED_WARPS) * sp, g_first1, (fp + g_first1) & 15u,
                                   warp + TILED_WARPS < h, nbytes, lane);
                    r0.sh = (r0.s_chunk & 3u) * 8u; r0.s_chunk &= ~3u;
                    r1.sh = (r1.s_chunk & 3u) * 8u; r1.s_chunk &= ~3u;
                    ragged = __any_sync(0xffffffffu, r0.do_byte || r1.do_byte);
                }
                mbar_wait(sm.full + 8 * ring.slot, ring.phase, __LINE__);
                const uint32_t box = sm.base + ring.slot * a.box_bytes;
                copy_out(r0, box, ragged, frame);
                copy_out(r1, box, ragged, frame);
                __syncwarp();
                if (lane == 0) mbar_arrive(sm.empty + 8 * ring.slot);
                ring.advance(stages);
            }
            continue;
        }

        const uint32_t g_row0 = g_cell + (uint32_t)warp * (uint32_t)a.dst_pitch;
        int n_ov = 0;
        uint32_t ov_sp0 = 0, ov_sp1 = 0;
        bool zero_base = false;
        if (BANDS && tile.cls == MCS_TILE_BAND) {
            // ---- BAND cell: its overlay descriptors into the overlay buffer, the overlay layers' box pitches ----
            n_ov = (tile.reserved >> 24) & 15;
            zero_base = ((tile.reserved >> 28) & 1) != 0;
            const uint32_t ov_full = sm.ov + a.ov_bytes, ov_empty = ov_full + 8;
            const int band_seq = (int)lds32(ov_full + 16 + 4 * warp);
            if (tid == 0) {
                if (band_seq > 0) mbar_wait(ov_empty, (uint32_t)((band_seq - 1) & 1), __LINE__);   // every warp is done with the last one
                mbar_expect_tx(ov_full, (uint32_t)n_ov * (MCS_CELL_W * MCS_CELL_H * 4u));
                bulk_g2s(sm.ov, a.band_desc + (size_t)id * (MCS_BAND_MAX_OVERLAYS * MCS_CELL_W * MCS_CELL_H),
                         (uint32_t)n_ov * (MCS_CELL_W * MCS_CELL_H * 4u), ov_full);
            }
            const int4 r0 = __ldg(a.band_issue + id * (1 + MCS_BAND_MAX_OVERLAYS) + 1);
            const int4 r1 = __ldg(a.band_issue + id * (1 + MCS_BAND_MAX_OVERLAYS) + 2);
            ov_sp0 = (uint32_t)a.layer_sp[r0.x];
            ov_sp1 = r1.x >= 0 ? (uint32_t)a.layer_sp[r1.x] : 0u;
            mbar_wait(ov_full, (uint32_t)(band_seq & 1), __LINE__);
            __syncwarp();
            if (lane == 0) sts32(ov_full + 16 + 4 * warp, (uint32_t)(band_seq + 1));
        }
        if (C == 3 && tile.cls == MCS_TILE_FAST && a.use_fast) {
            // ---- FAST cell: this thread's two group descriptors and its share of the warp's general list ----
            const uint32_t grp = rec + MCS_FAST_HEADER_BYTES;
            const uint32_t lst = rec + MCS_FAST_HEADER_BYTES + MCS_FAST_GROUP_BYTES;
            const uint2 w0 = lds64(grp + (warp * 32 + lane) * 8), w1 = lds64(grp + ((TILED_WARPS + warp) * 32 + lane) * 8);
            const int n_pass = ((int)lds8(rec + 32 + warp) + 31) >> 5;
            GenDesc gen[MCS_FAST_MAX_PASSES];
#pragma unroll
            for (int p = 0; p < MCS_FAST_MAX_PASSES; ++p) {
                uint2 e = make_uint2(0u, 0xffffffffu);
                if (p < n_pass) e = lds64(lst + ((p * TILED_WARPS + warp) * 32 + lane) * 8);
                gen[p] = expand_gen(e, lane);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(rec_release);
            const GroupDesc g0 = expand_group(w0), g1 = expand_group(w1);
            // one call per frame when the frame stride moves the rows' 16-byte phase
            const int n_call = phase_moves ? n_fr : 1, fr_call = phase_moves ? 1 : n_fr;
#define MCS_FAST_FRAMES(SP_)                                                                                        \
    for (int q = 0; q < n_call; ++q)                                                                                  \
        fast_frames<SP_>(a, g0, g1, gen, n_pass, sp, sm, ring, frame0 + (long long)q * a.dst_frame_stride, g_row0,     \
                         fr_call, c0, nbytes, h, warp, lane)
            if (sp == 512) MCS_FAST_FRAMES(512); else MCS_FAST_FRAMES(0);
#undef MCS_FAST_FRAMES
            continue;
        }

        // ---- WARP cell: expand this thread's plan-time pixel descriptors ----
        PxDesc d[8];
        {
            const uint32_t dp = rec + MCS_FAST_HEADER_BYTES + (warp * 32 + lane) * 4;
            uint32_t w[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) w[j] = lds32(dp + j * (TILED_WARPS * 32 * 4));
            __syncwarp();
            if (lane == 0) mbar_arrive(rec_release);
#pragma unroll
            for (int j = 0; j < 8; ++j) d[j] = expand_desc(w[j]);
        }
        uint32_t groups = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int row = warp + TILED_WARPS * (j >> 2), g0c = 32 * (j & 3);
            if (row < h && g0c < c1 && g0c + 32 > c0) groups |= 1u << j;
        }
        // the common box pitch of this channel count at compile time (128 columns at about unit scale), any other at run time
        constexpr int SP_MAIN = C == 1 ? 256 : C == 3 ? 512 : 640;
#define MCS_WARP_FRAMES(SP_, BAND_)                                                                                 \
    warp_frames<C, SP_, BAND_>(a, d, groups, sp, sm, ring, frame0, g_row0, n_fr, c0, nbytes, h, warp, lane, n_ov,     \
                               ov_sp0, ov_sp1, zero_base)
        if (BANDS && tile.cls == MCS_TILE_BAND) {
            MCS_WARP_FRAMES(0, BANDS);
            __syncwarp();
            if (lane == 0) mbar_arrive(sm.ov + a.ov_bytes + 8);   // done with the overlay descriptors
        } else {
            if (sp == SP_MAIN) MCS_WARP_FRAMES(SP_MAIN, false); else MCS_WARP_FRAMES(0, false);
        }
#undef MCS_WARP_FRAMES
    }
}

// ---- host side -----------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// Overlay-descriptor buffer of the BAND tiles (feather mode, fused form); 0 when the plan has none.
static size_t tiled_ov_bytes(const mcs_plan* plan) {
    return plan->band_fused && plan->n_band > 0 ? (size_t)plan->band_max_ov * MCS_CELL_W * MCS_CELL_H * 4 : 0;
}

static size_t tiled_smem_bytes(const mcs_plan* plan, int stages) {
    const int out_pitch = MCS_CELL_W * plan->channels + 16;
    return (size_t)stages * plan->box_bytes + 2 * TILED_MAX_STAGES * sizeof(uint64_t) + TILED_SCHED_BYTES +
           64 /* chunk-record barriers */ + (size_t)MCS_CELL_H * out_pitch + 16 + 2 * TILED_DESC_BUF_BYTES + 1024 +
           (tiled_ov_bytes(plan) ? tiled_ov_bytes(plan) + 64 : 0);
}

// Ring depth: as deep as fits a per-CTA budget that still leaves TILED_MIN_CTAS CTAs per SM.
static int tiled_stages(const mcs_plan* plan) {
    const size_t budget = (size_t)TILED_SMEM_BUDGET_KB * 1024;
    int s = TILED_MAX_STAGES;
    while (s > 3 && tiled_smem_bytes(plan, s) > budget) --s;
    return s;
}

const char* mcs_tiled_blocker(const mcs_plan* plan, const uint8_t* const* src, const int64_t* pitch,
                              const int64_t* fstride, int n_frames, int64_t dst_pitch) {
    if (!plan->tiled_ok) return plan->tiled_why;
    if (dst_pitch <= 0 || (long long)plan->out_h * dst_pitch >= (1ll << 32))
        return "output frame of 4 GiB or more (the tiled kernel addresses a frame with 32-bit offsets)";
    if (!get_encode_fn()) return "cuTensorMapEncodeTiled unavailable";
    if (plan->rows_need_pad && !plan->pad_promised)
        return "a source row is not a multiple of 4 bytes (zero-padded rows were not promised)";
    for (int k = 0; k < plan->n_layers; ++k) {
        if (pitch[k] < (((int64_t)plan->layers[k].src_w * plan->channels + 3) & ~(int64_t)3))
            return "source pitch smaller than the row rounded up to 4 bytes";
        if ((reinterpret_cast<uintptr_t>(src[k]) & 15) != 0) return "source base not 16-byte aligned";
        if ((pitch[k] & 15) != 0) return "source pitch not a multiple of 16 bytes";
        if (n_frames > 1 && (fstride[k] & 15) != 0) return "source frame stride not a multiple of 16 bytes";
        if (n_frames > 1 && fstride[k] <= 0) return "non-positive source frame stride";
    }
    return nullptr;
}

int mcs_launch_tiled(mcs_plan* plan, const uint8_t* const* src, const int64_t* pitch, const int64_t* fstride,
                     int n_frames, uint8_t* dst, int64_t dst_pitch, int64_t dst_frame_stride,
                     cudaStream_t stream) {
    TiledArgs a;
    memset(&a, 0, sizeof(a));
    bool hit = plan->cache_valid && plan->cache_frames == n_frames;
    for (int k = 0; hit && k < plan->n_layers; ++k)
        hit = plan->cache_src[k] == src[k] && plan->cache_pitch[k] == pitch[k] &&
              (n_frames == 1 || plan->cache_fstride[k] == fstride[k]);
    CUtensorMap* cache = reinterpret_cast<CUtensorMap*>(
        (reinterpret_cast<uintptr_t>(plan->tmap_cache) + 63) & ~(uintptr_t)63);
    if (!hit) {
        EncodeTiledFn enc = get_encode_fn();
        for (int k = 0; k < plan->n_layers; ++k) {
            const McsLayer& L = plan->layers[k];
            const cuuint64_t dims[3] = {(cuuint64_t)((L.src_w * plan->channels + 3) / 4), (cuuint64_t)L.src_h,
                                        (cuuint64_t)n_frames};
            const cuuint64_t strides[2] = {(cuuint64_t)pitch[k],
                                           (cuuint64_t)(n_frames > 1 ? fstride[k] : pitch[k] * L.src_h)};
            const cuuint32_t box[3] = {(cuuint32_t)L.bw4, (cuuint32_t)L.bh, 1u};
            const cuuint32_t estr[3] = {1u, 1u, 1u};
            CUresult r = enc(&cache[k], CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t*>(src[k]), dims,
                             strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) {
                mcs_set_error("mcs_stitch_u8: cuTensorMapEncodeTiled failed for layer %d (CUresult %d)", k, (int)r);
                plan->cache_valid = 0;
                return MCS_ERR_CUDA;
            }
            plan->cache_src[k] = src[k];
            plan->cache_pitch[k] = pitch[k];
            plan->cache_fstride[k] = n_frames > 1 ? fstride[k] : 0;
        }
        plan->cache_frames = n_frames;
        plan->cache_valid = 1;
    }
    for (int k = 0; k < plan->n_layers; ++k) a.tmap[k] = cache[k];
    a.tiles = plan->d_tiles;
    a.issue = plan->d_issue;
    a.layers = plan->d_layers;
    for (int k = 0; k < plan->n_layers; ++k) {
        a.layer_sp[k] = plan->layers[k].bw4 * 4;
        a.layer_ox[k] = plan->layers[k].ox;
    }
    a.desc = plan->d_desc;
    a.dst = dst;
    a.dst_pitch = dst_pitch;
    a.dst_frame_stride = dst_frame_stride;
    a.box_bytes = plan->box_bytes;
    a.stages = tiled_stages(plan);

    const size_t smem = tiled_smem_bytes(plan, a.stages);
    const bool bands = tiled_ov_bytes(plan) != 0;   // feather mode, fused form: the instantiation that knows BAND tiles
    void (*kern)(TiledArgs) = plan->channels == 1   ? (bands ? mcs_stitch_tiled_kernel<1, true> : mcs_stitch_tiled_kernel<1, false>)
                              : plan->channels == 3 ? (bands ? mcs_stitch_tiled_kernel<3, true> : mcs_stitch_tiled_kernel<3, false>)
                                                    : (bands ? mcs_stitch_tiled_kernel<4, true> : mcs_stitch_tiled_kernel<4, false>);
    {
        // The dynamic shared-memory limit is an attribute of the kernel (per device), not of the
        // plan: several plans with different box sizes share it, so it is only ever raised.
        static int attr_smem[64][6];   // [device][channel variant x BAND variant], bytes granted so far
        int dev = 0;
        MCS_CHECK_CUDA(cudaGetDevice(&dev));
        int& granted = attr_smem[dev & 63][(plan->channels == 1 ? 0 : plan->channels == 3 ? 1 : 2) + (bands ? 3 : 0)];
        if ((int)smem > granted) {
            MCS_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            granted = (int)smem;
        }
    }
    if (!plan->grid_ctas_per_sm) {
        int per_sm = 0, n_sm = 0, dev = 0;
        MCS_CHECK_CUDA(cudaGetDevice(&dev));
        MCS_CHECK_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
        MCS_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TILED_CTA_THREADS, smem));
        if (per_sm < 1) {
            mcs_set_error("mcs_stitch_u8: tiled kernel does not fit (smem %zu bytes)", smem);
            return MCS_ERR_UNSUPPORTED;
        }
        plan->grid_ctas_per_sm = per_sm;
        plan->n_sm = n_sm;
    }
    // Frame blocks: the CTAs sweep the tile table once per block of `frame_block` frames, so that at
    // any time they all work on the same few frames (few DRAM pages open at once, box overlaps of
    // neighbouring cells still in L2).
    const int fb = plan->frame_block < n_frames ? plan->frame_block : n_frames;
    a.frame_block = fb;
    a.n_blocks = (n_frames + fb - 1) / fb;
    a.nf_last = n_frames - (a.n_blocks - 1) * fb;

    long long grid = (long long)plan->n_sm * plan->grid_ctas_per_sm;
    const long long units = (long long)plan->n_tiles * fb;
    if (grid > units) grid = units;
    a.n_tiles = plan->n_tiles;
    // split the last resampled tiles of the sweep (about two per CTA) into four chunks each
    a.split_end = plan->class_first[MCS_SEG(MCS_TILE_COPY)];   // BAND, FAST and WARP tiles are the resampled ones
    a.split = fb >= 16 ? 4 : 1;
    const int split_tiles = 2 * (int)grid;
    {
        const char* env = getenv("MCS_TILED_SPLIT");   // tests: split factor (0 / 1 = no split)
        if (env) a.split = atoi(env) > 1 && fb >= atoi(env) ? atoi(env) : 1;
    }
    // A last frame block shorter than the split factor would cut its split tiles into chunks WITHOUT frames, each a
    // claim and a record copy for no work: no split then.
    if (a.split > 1 && a.nf_last < a.split) a.split = 1;
    a.split_first = a.split > 1 ? (a.split_end > split_tiles ? a.split_end - split_tiles : 0) : a.split_end;
    a.chunks_per_block = plan->n_tiles + (a.split_end - a.split_first) * (a.split - 1);
    {
        // one COPY / ZERO tile after every light_every - 1 resampled chunks, as long as both kinds last
        const int n_light = plan->n_tiles - a.split_end, n_heavy = a.chunks_per_block - n_light;
        a.n_heavy = n_heavy;
        a.light_every = n_light > 0 ? n_heavy / n_light + 1 : 2;
        if (a.light_every < 2) a.light_every = 2;
        int zone = n_light < n_heavy / (a.light_every - 1) ? n_light : n_heavy / (a.light_every - 1);   // light tiles placed
        a.light_end = zone * a.light_every;
        a.heavy_end = n_heavy + a.light_end / a.light_every;
    }
    if ((long long)a.n_blocks * a.chunks_per_block >= (1ll << 30)) {
        mcs_set_error("mcs_stitch_u8: %d frame blocks x %d chunks exceed the chunk counter", a.n_blocks, a.chunks_per_block);
        return MCS_ERR_UNSUPPORTED;
    }
    a.n_chunks = a.n_blocks * a.chunks_per_block;
    // chunks per claim: short chunks (few frames per launch) are claimed several at a time, so that a claim - one
    // atomic round trip of the producer thread - covers about 32 units of work, but never so many that the
    // CTAs could not all be served
    {
        int claim = 32 / fb;
        const long long fair = a.n_chunks / (4 * grid);
        if (claim > fair) claim = (int)fair;
        a.claim = claim < 1 ? 1 : claim > 8 ? 8 : claim;
    }
    a.work = plan->d_work;
    for (int c = 0; c <= MCS_N_CLASSES; ++c) a.class_first[c] = plan->class_first[c];
    a.band_issue = plan->d_band_issue;
    a.band_desc = plan->d_band_desc;
    a.feather_log2 = plan->feather_log2;
    a.ov_bytes = (int)tiled_ov_bytes(plan);
    a.fast = plan->d_fast;
    a.fast_stride = plan->fast_stride;
    a.fast_passes = plan->fast_passes;
    // the group path stores whole words into the staging rows, which carry the 16-byte phase of the
    // output rows: every output row of every frame must start on a 4-byte boundary
    a.use_fast = plan->d_fast != nullptr && (reinterpret_cast<uintptr_t>(dst) & 3) == 0 && (dst_pitch & 3) == 0 &&
                 (n_frames == 1 || (dst_frame_stride & 3) == 0);
    kern<<<(unsigned)grid, TILED_CTA_THREADS, smem, stream>>>(a);
    mcs_count_launch(1);
    MCS_CHECK_CUDA(cudaGetLastError());
    return MCS_OK;
}
