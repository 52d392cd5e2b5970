// Internal definitions shared by the translation units of libmcs_b200.so.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdarg.h>
#include <stdio.h>

#include "mcs.h"

#define MCS_ABI_VERSION 3

// ---- error plumbing -------------------------------------------------------
void mcs_set_error(const char* fmt, ...);
void mcs_count_launch(int n);

#define MCS_CHECK_ARG(cond, ...)                 \
    do {                                         \
        if (!(cond)) {                           \
            mcs_set_error(__VA_ARGS__);          \
            return MCS_ERR_INVALID;              \
        }                                        \
    } while (0)

#define MCS_CHECK_CUDA(expr)                                                        \
    do {                                                                            \
        cudaError_t _e = (expr);                                                    \
        if (_e != cudaSuccess) {                                                    \
            mcs_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),   \
                          __FILE__, __LINE__);                                      \
            return MCS_ERR_CUDA;                                                    \
        }                                                                           \
    } while (0)

// ---- compositing plan -----------------------------------------------------
// One camera of the panorama, in the form the kernels consume (host copy in the plan, device
// copy in plan->d_layers).
struct McsLayer {
    double mi[9];            // inverse homography (layer canvas frame -> source), cv::invert closed form
    int rx0, ry0, rx1, ry1;  // visible rectangle, output coordinates, half open
    int px0, py0, px1, py1;  // the rectangle as it was PASTED (before any super-mode crop cut it): the feather
                             // blend measures its distances to these edges; equal to the visible rectangle
                             // unless mcs_plan_set_paste_rects says otherwise
    int ox, oy;              // origin of the layer's canvas frame in output coordinates
    int src_w, src_h;
    int kind;                // MCS_LAYER_*
    int affine;              // mi[6] == mi[7] == 0
    int bw4;                 // tiled variant: staged box width in 4-byte words (multiple of 4, <= 256)
    int bh;                  // tiled variant: staged box height in rows (<= 256)
    int w_safe;              // |W| stays in [1e-3, 1e6] with one sign over the rectangle: the
                             // branch-free division of the tiled kernel is exact there
    int map_w, map_h;        // REMAP layers: size of the coordinate map (= the layer's canvas frame)
    const int2* map;         // REMAP layers: device, map_h x map_w 1/32-px source coordinates (X, Y)
};

// Work item of the tiled kernel: the part of one 128 x 16 cell that one layer owns.  Cells sit on
// a grid anchored at panorama column 0 (cell column 0 at output x = 128*i).
struct McsTile {
    int cx0;         // output x of cell column 0
    int y0;          // output y of the first row
    short c0, c1;    // owned cell columns [c0, c1), 0 <= c0 < c1 <= 128
    short h;         // rows, 1..16
    short layer;     // owner layer, -1 for background
    short cls;       // MCS_TILE_*
    short flags;     // estimated cost of one frame of the tile (work-split weight)
    int bx;          // staged box origin: 4-byte word index within the source row (may be negative)
    int by;          // staged box origin: source row (may be negative)
    int reserved;    // bytes of the staged box (mbarrier transaction count)
};
static_assert(sizeof(McsTile) == 32, "McsTile must stay 32 bytes");

#define MCS_TILED_WARPS 8   // resampling warps of the tiled kernel; each owns two rows of a cell
#define MCS_CELL_W 128
#define MCS_CELL_H (2 * MCS_TILED_WARPS)

#define MCS_TILE_ZERO 0   // nothing to sample: write zeros
#define MCS_TILE_COPY 1   // verbatim paste of the source window
#define MCS_TILE_WARP 2   // fixed-point bilinear resample from the staged source box, one descriptor per pixel
#define MCS_TILE_FAST 3   // the same resample through the group descriptors (four adjacent pixels per thread share
                          // one source window; pixels that do not fit that template go through a short per-pixel list)
#define MCS_TILE_BAND 4   // feather mode: a resampled tile some of whose pixels blend with one or two outer layers
                          // (the seam band of a pasted rectangle); per frame it stages one box per layer involved
#define MCS_N_CLASSES 5
// The tile table is sorted by descending class; segment s of plan->class_first holds class MCS_N_CLASSES - 1 - s.
#define MCS_SEG(cls) (MCS_N_CLASSES - 1 - (cls))

// BAND tiles: at most this many outer layers blend into one tile (more -> the plan keeps the two-pass band path)
#define MCS_BAND_MAX_OVERLAYS 2
#define MCS_BAND_MAX_LOG2 5   // overlay weights (a + 1 <= 32) travel in 6 bits of the overlay descriptors

// Group ("fast") descriptors of a WARP tile, C == 3 only (mcs_tiles.cu builds them, mcs_stitch_tiled.cu reads them).
// One record per tile: [McsTile, 32 B][general-list length of each warp, 8 x u8][pad to 64 B]
// [group descriptors 2 slots x 8 warps x 32 lanes x uint2][general list: passes x 8 warps x 32 lanes x uint2].
#define MCS_FAST_HEADER_BYTES 64
#define MCS_FAST_GROUP_BYTES (2 * MCS_TILED_WARPS * 32 * 8)
#define MCS_FAST_PASS_BYTES (MCS_TILED_WARPS * 32 * 8)
#define MCS_FAST_MAX_PASSES 2

#define MCS_BOX_BYTES_MAX (40 * 1024)   // per staged source box

#define MCS_FRAME_BLOCK_DEFAULT 64

struct mcs_plan {
    int n_layers;
    int channels;
    int out_w, out_h;
    int device;
    McsLayer layers[MCS_MAX_LAYERS];
    int last_variant;
    int feather_log2;        // 0 = the reference's overwrite paste, > 0 = feather blend over 2^n pixels
    int4* d_strips;          // feather: band strips {x0, y0, x1, y1} inside the pasted rectangles
    long long* d_strip_prefix;   // n_strips + 1 running pixel counts
    int n_strips;
    long long strip_pixels;
    // feather: plan-time sample table of the band pixels (mcs_stitch.cu), nullptr = evaluate on the fly
    int2* d_band_xy;         // strip_pixels output coordinates
    unsigned char* d_band_cnt;   // samples per band pixel (<= n_layers)
    int4* d_band_ent;        // [n_layers][strip_pixels] {X, Y, layer, weight of the value so far}
    int force_variant;       // 0 = automatic, 1 = gather, 2 = tiled (diagnostics)
    // tiled variant
    int tiled_ok;            // tile table built and every box within limits
    int rows_need_pad;       // some source row is not a multiple of 4 bytes: the tiled variant then needs
    int pad_promised;        // the caller's promise that rows are followed by zero bytes up to one (mcs.h)
    char tiled_why[160];     // why not, when tiled_ok == 0
    int n_tiles;
    int box_bytes;           // shared-memory bytes of one staging buffer (max over layers, 128-aligned)
    McsTile* d_tiles;
    int4* d_issue;           // per tile {layer, bx, by, staged box bytes}: what the box issuer of the tiled kernel reads
    McsLayer* d_layers;
    int2* d_maps[MCS_MAX_LAYERS];   // coordinate maps of the REMAP layers (owned by the plan)
    uint32_t* d_desc;        // per-pixel descriptors of the WARP tiles, 2048 words per tile (mcs_tiles.cu)
    uint8_t* d_fast;         // group-descriptor records of the FAST tiles (they come first in the table), or nullptr
    int fast_stride;         // bytes per record: header + groups + fast_passes general passes
    int fast_passes;         // general passes every record carries (max over the FAST tiles, 0..MCS_FAST_MAX_PASSES)
    int src_win[MCS_MAX_LAYERS][4];   // per layer: source window {x0, y0, x1, y1} its owned pixels read
    int src_win_valid;       // set with the tile table; otherwise the whole frame counts
    int* h_row_span[MCS_MAX_LAYERS];   // host, per source row {x0, x1} of the pixels read (nullptr = unknown)
    int frame_block;         // frames per sweep of the tile table (mcs_launch_tiled)
    // cache of the TMA descriptors of the last call (keyed by the source table)
    unsigned char tmap_cache[MCS_MAX_LAYERS * 128 + 64];
    const void* cache_src[MCS_MAX_LAYERS];
    long long cache_pitch[MCS_MAX_LAYERS];
    long long cache_fstride[MCS_MAX_LAYERS];
    int cache_frames;
    int cache_valid;
    int grid_ctas_per_sm;    // resident CTAs per SM of the tiled kernel (0 = not queried yet)
    int n_sm;
    // Work split of the tiled kernel: the CTAs claim chunks (a tile for one block of frames) at run time from
    // d_work[0]; d_work[1] counts finished CTAs and the last one rewinds both, so a plan serves ONE launch at a
    // time (one stream), see mcs.h.
    int class_first[MCS_N_CLASSES + 1];   // the tile table is sorted BAND, FAST, WARP, COPY, ZERO: first tile of
                             // each class, then n_tiles
    // feather mode, fused form (mcs_tiles.cu): BAND tiles are the first n_band tiles of the table
    int band_fused;          // the tiled kernel blends the seam bands itself (no second pass)
    int blend_custom;        // weight maps or cut (super-mode) rectangles: only the fused form computes them
    int n_band;
    int band_max_ov;         // most outer layers any BAND tile blends with (sizes the kernel's overlay buffer)
    int4* d_band_issue;      // [n_band][1 + MCS_BAND_MAX_OVERLAYS] {layer, bx, by, box bytes | n_overlays << 24}
    uint32_t* d_band_desc;   // [n_band][MCS_BAND_MAX_OVERLAYS][2048] overlay descriptors: per-pixel descriptor of the
                             // outer layer | weight of the value so far << 26 (0 = pixel not blended with this layer)
    uint8_t* d_wmap[MCS_MAX_LAYERS];   // per layer k >= 1: weight map of the paste of stage k (over the pasted
                             // rectangle of layer k - 1, values 0 .. 2^feather_log2), nullptr = the distance ramp
    unsigned* d_work;
    // camera-weighted blend (mcs_plan_set_camera_weights, mcs_stitch_weighted.cu)
    int cw_active;           // the plan blends every camera that sees a pixel, normalised by the summed weights
    uint8_t* d_cwmap[MCS_MAX_LAYERS];   // per layer: device weight map, src_h x src_w bytes (nullptr = 255 everywhere)
    long long cw_contrib[MCS_MAX_LAYERS];   // per layer: output pixels it contributes to
    int cw_maps;             // the maps of the last mcs_plan_set_camera_weights are held: also when the rig was refused
                             // for the camera-weighted kernel (more than MCS_CW_MAX_CONTRIB contributors), since the
                             // multi-band blend takes such rigs
    // multi-band blend (mcs_plan_set_multiband, mcs_stitch_multiband.cu)
    int mb_on;               // the multi-band blend serves the plan
    int mb_bands;            // its effective band count (clamped like MultiBandBlender::prepare)
    struct McsMultiband* mb; // geometry, weight pyramids and workspace
};


// 3x3 float64 inverse with cv::invert's association (host, no FMA contraction).
bool mcs_invert3x3(const double* m, double* out);

// Builds the tile table of the tiled variant (mcs_tiles.cu).  Never fails the plan: on any
// problem it leaves tiled_ok = 0 with the reason in tiled_why and the gather variant is used.
void mcs_plan_build_tiles(mcs_plan* plan);
void mcs_plan_free_tiles(mcs_plan* plan);

// Feather mode: builds / frees the plan-time sample table of the band pixels (mcs_stitch.cu).  A
// failure to build leaves the table empty; the on-the-fly band kernel then serves the mode.
void mcs_feather_build_table(mcs_plan* plan);
void mcs_feather_free_table(mcs_plan* plan);

// Camera-weighted blend (mcs_stitch_weighted.cu): at most this many cameras blend into one pixel (their
// weights stay in registers, and the multiply-high division is exact for sums up to 4 * 255)
#define MCS_CW_MAX_CONTRIB 4
// Per layer, the output pixels it contributes to, and the most contributors of any pixel (synchronous).
int mcs_camera_weights_count(const mcs_plan* plan, long long* contrib, int* max_count);
int mcs_launch_weighted(const mcs_plan* plan, const uint8_t* const* src, const int64_t* pitch,
                        const int64_t* fstride, int n_frames, uint8_t* dst, int64_t dst_pitch,
                        int64_t dst_frame_stride, cudaStream_t stream);

// Multi-band blend (mcs_stitch_multiband.cu): at most this many pyramid levels (8 bands + the top)
#define MCS_MB_MAX_LEVELS 9
// Builds the geometry, the weight pyramids and sums of the plan's held camera maps and the workspace for
// `bands` requested bands (synchronous); frees them.
int mcs_multiband_build(mcs_plan* plan, int bands);
void mcs_multiband_free(mcs_plan* plan);
int mcs_launch_multiband(const mcs_plan* plan, const uint8_t* const* src, const int64_t* pitch, const int64_t* fstride,
                         int n_frames, uint8_t* dst, int64_t dst_pitch, int64_t dst_frame_stride, cudaStream_t stream);

// Tiled variant (mcs_stitch_tiled.cu): why it cannot serve a call (nullptr = it can), and its launch.
const char* mcs_tiled_blocker(const mcs_plan* plan, const uint8_t* const* src, const int64_t* pitch,
                              const int64_t* fstride, int n_frames, int64_t dst_pitch);
int mcs_launch_tiled(mcs_plan* plan, const uint8_t* const* src, const int64_t* pitch, const int64_t* fstride,
                     int n_frames, uint8_t* dst, int64_t dst_pitch, int64_t dst_frame_stride,
                     cudaStream_t stream);
